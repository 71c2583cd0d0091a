"""torch.autograd wrappers around the libb2nerf.so kernels.

Every op takes/returns contiguous fp32 CUDA tensors on the current stream;
``custom_fwd(cast_inputs=float32)`` makes them safe under the
``torch.amp.autocast('cuda')`` regions of run.py:1092,1818.
"""
from __future__ import annotations

import ctypes
import math
from typing import List, Optional, Sequence

import numpy as np
import torch
from torch.amp import custom_bwd, custom_fwd

from . import _lib
from ._lib import HashLevelC, current_rows, ptr, require_cuda, stream, with_ctx_rows

# hash_encode sorts its points into spatial order (b2n_hash_order) from this many points on, when the input needs no
# gradient and the F = 2 pair-lane kernels run: measured to pay at C2's 24 M points; smaller sets are not sorted
HASH_ORDER_MIN_POINTS = 1 << 23


def call(name, *args, work=(0.0, 0.0)):
    _lib.call(name, *args, work=work)        # late-bound so that _lib.PROFILER can be swapped at run time

ACT_NONE, ACT_RELU, ACT_SIGMOID = 0, 1, 2
_ACT = {"none": ACT_NONE, "relu": ACT_RELU, "sigmoid": ACT_SIGMOID}


def _narrow_out(*shape, device, dtype=torch.float32):
    """Point-indexed tensors of a few floats per row (rgb, sigma, delta_x and their gradients).  With a device-side row
    count the rows behind it are never written by the kernels, but torch-side reductions over rows exist downstream
    (``displacement_scale.grad = sum(g * y)``): those rows must hold zeros, not whatever the allocator returns."""
    if current_rows() is not None:
        return torch.zeros(*shape, device=device, dtype=dtype)
    return torch.empty(*shape, device=device, dtype=dtype)


def _c(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# ----------------------------------------------------------------------------
# hash-grid geometry (host side; passed by value to the kernels)
# ----------------------------------------------------------------------------

_libm = ctypes.CDLL("libm.so.6")
for _fn in ("exp2f", "log2f", "ceilf"):
    getattr(_libm, _fn).restype = ctypes.c_float
    getattr(_libm, _fn).argtypes = [ctypes.c_float]


class HashGeometry:
    """Per-level scale / resolution / size / offset of a tinycudann-style HashGrid
    (semantics: SURVEY.md 8a/A2).  Computed once on the host in fp32 with libm,
    like upstream does, and handed to every kernel call so that host and device
    can never disagree on a resolution."""

    def __init__(self, n_levels: int, base_resolution: int, per_level_scale: float, log2_hashmap_size: int,
                 n_features: int = 2):
        if not (1 <= n_levels <= 32):
            raise ValueError("n_levels must be in [1, 32]")
        if n_features not in (1, 2, 4):
            raise ValueError("n_features_per_level must be 1, 2 or 4")
        self.n_levels, self.n_features = n_levels, n_features
        log2s = _libm.log2f(ctypes.c_float(per_level_scale))
        arr = (HashLevelC * n_levels)()
        offset = 0
        self.levels = []
        for l in range(n_levels):
            e = float(np.float32(np.float32(l) * np.float32(log2s)))
            scale = np.float32(np.float32(_libm.exp2f(ctypes.c_float(e))) * np.float32(base_resolution)) - np.float32(1.0)
            res = int(_libm.ceilf(ctypes.c_float(float(scale)))) + 1
            dense = res ** 3
            size = min((min(dense, (1 << 31) - 1) + 7) // 8 * 8, 1 << log2_hashmap_size)
            hashed = size < dense
            arr[l] = HashLevelC(float(scale), res, size, offset, int(hashed))
            self.levels.append((float(scale), res, size, offset, hashed))
            offset += size
        self.c_levels = arr
        self.n_entries = offset
        self.n_params = offset * n_features
        self.out_dim = n_levels * n_features


class _HashEncode(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, table, geom: HashGeometry, bound: float, sink):
        require_cuda(x, table)
        ctx.rows = current_rows()
        x, table = _c(x), _c(table)
        if x.dim() != 2 or x.shape[1] != 3:
            raise ValueError("hash_encode expects x of shape [P, 3]")
        if table.numel() != geom.n_params:
            raise ValueError(f"hash table has {table.numel()} params, geometry needs {geom.n_params}")
        Pn = x.shape[0]
        out = torch.empty(Pn, geom.out_dim, device=x.device, dtype=torch.float32)
        work = (Pn * (12 + geom.n_levels * geom.n_features * 4 * 9), 0.0)
        ctx.order = None
        if Pn >= HASH_ORDER_MIN_POINTS and geom.n_features == 2 and not ctx.needs_input_grad[0] and _lib.hash_config()[0] == 3:
            # spatial order (b2n_hash_order): the warps of both kernels hold nearby points; features are unchanged
            order = torch.empty(Pn, device=x.device, dtype=torch.int32)
            xs = torch.empty_like(x)
            scratch = torch.empty(_lib.lib.b2n_hash_order_scratch(Pn) // 4, device=x.device, dtype=torch.int32)
            call("b2n_hash_order", ptr(x), Pn, float(bound), ptr(order), ptr(xs), ptr(scratch), stream(),
                 work=(Pn * (12 + 4 + 4 + 12 + 4 + 12), 0.0))
            call("b2n_hash_fwd_ordered", ptr(xs), ptr(order), Pn, float(bound), ptr(table), geom.c_levels, geom.n_levels,
                 geom.n_features, ptr(out), geom.out_dim, 0, stream(), work=work)
            x, ctx.order = xs, order
        else:
            call("b2n_hash_fwd", ptr(x), Pn, float(bound), ptr(table), geom.c_levels, geom.n_levels, geom.n_features,
                 ptr(out), geom.out_dim, 0, stream(), work=work)
        ctx.save_for_backward(x, table)
        ctx.geom, ctx.bound = geom, bound
        ctx.sink = sink if (sink is not None and ctx.needs_input_grad[1]) else None
        if ctx.sink is not None:
            ctx.sink.uses += 1
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g):
        x, table = ctx.saved_tensors
        geom = ctx.geom
        g = _c(g)
        need_x, need_t = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        g_x = torch.empty_like(x) if need_x else None
        Pn, L, F = x.shape[0], geom.n_levels, geom.n_features
        bytes_t = (12 + L * F * 4 * 17) * int(need_t)
        bytes_x = (24 + L * F * 4 * 9) * int(need_x)

        def launch(g_table, gx, lo, hi, nbytes):
            if ctx.order is not None:             # x is in sorted order (forward); no input gradient on this path
                call("b2n_hash_bwd_ordered", ptr(x), ptr(ctx.order), Pn, float(ctx.bound), ptr(table), geom.c_levels, L,
                     F, ptr(g), geom.out_dim, 0, ptr(g_table), lo, hi, stream(), work=(Pn * nbytes, 0.0))
                return
            call("b2n_hash_bwd", ptr(x), Pn, float(ctx.bound), ptr(table), geom.c_levels, L, F, ptr(g), geom.out_dim, 0,
                 ptr(g_table), ptr(gx), 0, lo, hi, stream(), work=(Pn * nbytes, 0.0))

        sink = ctx.sink
        if sink is None or not need_t:
            g_table = torch.zeros_like(table) if need_t else None
            if need_x or need_t:
                launch(g_table, g_x, 0, -1, bytes_t + bytes_x)
            return g_x, g_table, None, None, None
        # data-parallel direct path: accumulate into the flat gradient buffer; the last backward of the step scatters
        # the fine levels first and hands their (contiguous, level-major) slice to the reducer while the coarse levels
        # are still being scattered
        sink.uses -= 1
        last = sink.uses <= 0
        split = sink.split_level if (last and F == 2 and 0 < sink.split_level < L and sink.split_level % 4 == 0) else 0
        if split:
            cut = geom.levels[split][3] * F                   # first element of level `split`
            launch(sink.view, None, split, L, bytes_t * (L - split) / L)
            sink.on_ready(sink, cut, sink.view.numel())
            launch(sink.view, g_x, 0, split, bytes_t * split / L + bytes_x)
            sink.on_ready(sink, 0, cut)
        else:
            launch(sink.view, g_x, 0, -1, bytes_t + bytes_x)
            if last:
                sink.on_ready(sink, 0, sink.view.numel())
        return g_x, None, None, None, None


def hash_encode(x, table, geom: HashGeometry, bound: float):
    """x [P,3] world coords (bound > 0) or unit-cube coords (bound == 0) -> [P, L*F]."""
    sink = getattr(table, "_b2n_grad_sink", None) if torch.is_grad_enabled() else None
    return _HashEncode.apply(x, table, geom, bound, sink)


class _HashTriBlend(torch.autograd.Function):
    """sum_i w_i(t) * HashGrid_i(x) over the start / mid / end deformation grids of Part 4 (src/core.py:308-335):
    one kernel forward (b2n_hash_tri_fwd), one backward (b2n_hash_tri_bwd)."""

    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, t, t0, t1, t2, geom: HashGeometry, bound: float, sinks):
        require_cuda(x, t, t0, t1, t2)
        ctx.rows = current_rows()
        # data-parallel direct path (b2n.dp.GradSink, see _HashEncode): per-table in-place accumulation
        ctx.sinks = [sk if (sk is not None and ctx.needs_input_grad[2 + i]) else None for i, sk in enumerate(sinks)]
        for sk in ctx.sinks:
            if sk is not None:
                sk.uses += 1
        x, t, t0, t1, t2 = _c(x), _c(t).reshape(-1), _c(t0), _c(t1), _c(t2)
        if geom.n_features != 2:
            raise ValueError("hash_tri_blend needs 2 features per level")
        if t.shape[0] != x.shape[0] or any(tb.numel() != geom.n_params for tb in (t0, t1, t2)):
            raise ValueError("hash_tri_blend: one time per point and three tables of the shared geometry")
        Pn = x.shape[0]
        out = torch.empty(Pn, geom.out_dim, device=x.device)
        call("b2n_hash_tri_fwd", ptr(x), ptr(t), Pn, float(bound), ptr(t0), ptr(t1), ptr(t2), geom.c_levels,
             geom.n_levels, ptr(out), geom.out_dim, stream(),
             work=(Pn * (16 + geom.n_levels * 2 * 4 * (2 * 8 + 1)), 0.0))
        ctx.save_for_backward(x, t)
        ctx.geom, ctx.bound, ctx.shapes = geom, bound, (t0.shape, t1.shape, t2.shape)
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g):
        x, t = ctx.saved_tensors
        geom = ctx.geom
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            raise RuntimeError("hash_tri_blend has no gradient w.r.t. positions or times")
        g = _c(g)
        sinks = ctx.sinks
        grads = [(sinks[i].view if sinks[i] is not None else torch.zeros(shape, device=x.device))
                 if ctx.needs_input_grad[2 + i] else None for i, shape in enumerate(ctx.shapes)]
        if any(gr is not None for gr in grads):
            call("b2n_hash_tri_bwd", ptr(x), ptr(t), x.shape[0], float(ctx.bound), geom.c_levels, geom.n_levels, ptr(g),
                 geom.out_dim, ptr(grads[0]), ptr(grads[1]), ptr(grads[2]), stream(),
                 work=(x.shape[0] * (16 + geom.n_levels * 2 * 4 * (1 + 2 * 2 * 8)), 0.0))
        for i, sk in enumerate(sinks):
            if sk is not None:
                sk.uses -= 1
                if sk.uses <= 0:
                    sk.on_ready(sk, 0, sk.view.numel())
                grads[i] = None                       # accumulated in place: nothing for autograd to add
        return None, None, grads[0], grads[1], grads[2], None, None, None


def hash_tri_blend(x, t, tables: Sequence[torch.Tensor], geom: HashGeometry, bound: float):
    """Tent-weighted blend of three hash grids sharing ``geom`` at per-point times t in [0, 1]: [P, L*2]."""
    on = torch.is_grad_enabled()
    return _HashTriBlend.apply(x, t, tables[0], tables[1], tables[2], geom, bound,
                               [getattr(tb, "_b2n_grad_sink", None) if on else None for tb in tables])


# ----------------------------------------------------------------------------
# Fourier features
# ----------------------------------------------------------------------------

class _Fourier(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, bands):
        require_cuda(x, bands)
        ctx.rows = current_rows()
        x, bands = _c(x), _c(bands)
        Pn, D = x.shape
        L = bands.numel()
        if D > 4:
            raise ValueError("fourier_encode supports input_dim <= 4")
        W = D + 2 * D * L
        out = torch.empty(Pn, W, device=x.device, dtype=torch.float32)
        call("b2n_pe_fwd", ptr(x), Pn, D, ptr(bands), L, ptr(out), W, 0, stream())
        ctx.save_for_backward(x, bands)
        return out

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g):
        if not ctx.needs_input_grad[0]:
            return None, None
        x, bands = ctx.saved_tensors
        g = _c(g)
        gx = torch.empty_like(x)
        call("b2n_pe_bwd", ptr(x), x.shape[0], x.shape[1], ptr(bands), bands.numel(), ptr(g), g.shape[1], 0,
             ptr(gx), 0, stream())
        return gx, None


def fourier_encode(x, bands):
    if bands.numel() == 0:
        return x
    return _Fourier.apply(x, bands)


# ----------------------------------------------------------------------------
# dense layers (fp32 exact path)
# ----------------------------------------------------------------------------

class _Linear(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x, W, b, act: int):
        require_cuda(x, W, b)
        if current_rows() is not None:
            raise RuntimeError("the fp32 layer-by-layer path does not support a device-side row count "
                               "(march(static=True)): use the 16-bit fused path (b2n.set_mlp_precision('bf16'))")
        x, W, b = _c(x), _c(W), _c(b)
        Pn, K = x.shape
        N = W.shape[0]
        if W.shape[1] < K:
            raise ValueError(f"linear: weight has {W.shape[1]} input columns, activations have {K}")
        y = torch.empty(Pn, N, device=x.device, dtype=torch.float32)
        # W may be wider than x (zero-padded FullyFusedMLP input columns): ldw = W.shape[1], K = x width
        call("b2n_linear_fwd", ptr(x), K, ptr(W), W.shape[1], ptr(b), ptr(y), N, Pn, K, N, act, stream(),
             work=(4.0 * Pn * (K + N), 2.0 * Pn * K * N))
        ctx.save_for_backward(x, W, y if act != ACT_NONE else None)
        ctx.act, ctx.has_b = act, b is not None
        return y

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, gy):
        x, W, y = ctx.saved_tensors
        Pn, K = x.shape
        N = W.shape[0]
        gy = _c(gy)
        if ctx.act != ACT_NONE:
            gy = gy.clone()
            call("b2n_act_bwd", ptr(gy), N, ptr(y), N, Pn, N, ctx.act, stream())
        gx = gW = gb = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(x)
            call("b2n_linear_dgrad", ptr(gy), N, ptr(W), W.shape[1], None, 0, ACT_NONE, ptr(gx), K, Pn, K, N, 0,
                 stream(), work=(4.0 * Pn * (K + N), 2.0 * Pn * K * N))
        if ctx.needs_input_grad[1]:
            gW = torch.zeros_like(W)
            gb = torch.zeros(N, device=x.device, dtype=torch.float32) if ctx.has_b and ctx.needs_input_grad[2] else None
            call("b2n_linear_wgrad", ptr(gy), N, ptr(x), K, ptr(gW), W.shape[1], ptr(gb), Pn, K, N, stream(),
                 work=(4.0 * Pn * (K + N), 2.0 * Pn * K * N))
        return gx, gW, gb, None


def linear(x, W, b=None, act: str = "none"):
    """act(x @ W[:, :x.shape[1]].T + b)"""
    return _Linear.apply(x, W, b, _ACT[act])


class _SigmaHead(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, h):
        require_cuda(h)
        if current_rows() is not None:
            raise RuntimeError("the fp32 layer-by-layer path does not support a device-side row count "
                               "(march(static=True)): use the 16-bit fused path (b2n.set_mlp_precision('bf16'))")
        h = _c(h)
        Pn = h.shape[0]
        sigma = torch.empty(Pn, 1, device=h.device, dtype=torch.float32)
        call("b2n_sigma_head_fwd", ptr(h), h.shape[1], Pn, ptr(sigma), stream())
        ctx.save_for_backward(h)
        return sigma

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, gs):
        h, = ctx.saved_tensors
        gh = torch.zeros_like(h)
        call("b2n_sigma_head_bwd", ptr(h), h.shape[1], h.shape[0], ptr(_c(gs)), ptr(gh), h.shape[1], stream())
        return gh


def sigma_head(h):
    """softplus(h[:, 0:1] - 5)   (src/decoders.py:153)"""
    return _SigmaHead.apply(h)


# ----------------------------------------------------------------------------
# compositing
# ----------------------------------------------------------------------------

class _Composite(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, rgb, sigma, dx, z, rays_d, bg, mask_words, ray_offset):
        require_cuda(rgb, sigma, z, rays_d)
        ctx.rows = current_rows()
        rgb, sigma, dx, z, rays_d, bg = _c(rgb), _c(sigma), _c(dx), _c(z), _c(rays_d), _c(bg)
        B, N = z.shape
        dev = z.device
        color = torch.empty(B, 3, device=dev)
        depth = torch.empty(B, device=dev)
        acc = torch.empty(B, device=dev)
        mdx = torch.empty(B, 3, device=dev) if dx is not None else None
        per_ray = int(bg is not None and bg.dim() == 2)
        if per_ray and bg.shape[0] != B:
            raise ValueError("bg_color must be [3] or [n_rays, 3]")
        call("b2n_composite_fwd", ptr(rgb), ptr(sigma), ptr(dx), ptr(z), ptr(rays_d), ptr(bg), per_ray,
             ptr(mask_words), ptr(ray_offset), B, N, ptr(color), ptr(depth), ptr(acc), ptr(mdx), stream(),
             work=(sigma.numel() * (16 + (12 if dx is not None else 0)) + 4.0 * B * N + 44.0 * B, 0.0))
        ctx.save_for_backward(rgb, sigma, dx, z, rays_d, bg, mask_words, ray_offset)
        ctx.per_ray = per_ray
        if mdx is None:
            mdx = torch.zeros(0, device=dev)
            ctx.mark_non_differentiable(mdx)
        return color, depth, acc, mdx

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g_color, g_depth, g_acc, g_mdx):
        rgb, sigma, dx, z, rays_d, bg, mask_words, ray_offset = ctx.saved_tensors
        B, N = z.shape
        g_rgb = _narrow_out(*rgb.shape, device=rgb.device)
        g_sigma = _narrow_out(*sigma.shape, device=rgb.device)
        g_dx = _narrow_out(*dx.shape, device=rgb.device) if dx is not None else None
        if dx is None:
            g_mdx = None
        call("b2n_composite_bwd", ptr(rgb), ptr(sigma), ptr(dx), ptr(z), ptr(rays_d), ptr(bg), ctx.per_ray,
             ptr(mask_words), ptr(ray_offset), B, N, ptr(_c(g_color)), ptr(_c(g_depth)), ptr(_c(g_acc)),
             ptr(_c(g_mdx)), ptr(g_rgb), ptr(g_sigma), ptr(g_dx), stream(),
             work=(sigma.numel() * (32 + (24 if dx is not None else 0)) + 4.0 * B * N + 32.0 * B, 0.0))
        return g_rgb, g_sigma, g_dx, None, None, None, None, None


def composite(rgb, sigma, z, rays_d, bg=None, dx=None, mask_words=None, ray_offset=None):
    """Alpha compositing of per-sample fields.  rgb [P,3], sigma [P] (or [P,1]),
    dx [P,3]|None in dense (P = B*N) or compact layout (mask_words/ray_offset given).
    Returns color [B,3], depth [B], acc [B], mean_dx [B,3] | None."""
    sigma = sigma.reshape(-1)
    rgb = rgb.reshape(-1, 3)
    if dx is not None:
        dx = dx.reshape(-1, 3)
    color, depth, acc, mdx = _Composite.apply(rgb, sigma, dx, z, rays_d, bg, mask_words, ray_offset)
    return color, depth, acc, (mdx if dx is not None else None)


# ----------------------------------------------------------------------------
# fused 64-wide Instant decoder (bf16 tensor cores)
# ----------------------------------------------------------------------------

_MLP_PRECISION = {"mode": "bf16"}


def set_mlp_precision(mode: str):
    """'bf16' (default): fused tensor-core decoder, 1e-2 parity class, like the reference's fp16 tinycudann nets.
    'fp32': layer-by-layer fp32 kernels, 1e-4 parity class."""
    if mode not in ("bf16", "fp32"):
        raise ValueError(mode)
    _MLP_PRECISION["mode"] = mode


def mlp_precision() -> str:
    return _MLP_PRECISION["mode"]


class _InstantMLP(torch.autograd.Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x_enc, dirs, bands, sigma_params, color_params, pad_value):
        require_cuda(x_enc, dirs, bands, sigma_params, color_params)
        ctx.pad_value = float(pad_value)
        ctx.rows = current_rows()
        x_enc, dirs, bands, sp, cp = _c(x_enc), _c(dirs), _c(bands), _c(sigma_params), _c(color_params)
        Pn, pos_dim = x_enc.shape
        rgb = _narrow_out(Pn, 3, device=x_enc.device)
        sigma = _narrow_out(Pn, 1, device=x_enc.device)
        flops = 2.0 * Pn * (64 * pos_dim + 16 * 64 + 64 * 43 + 64 * 64 + 3 * 64)
        call("b2n_instant_mlp_fwd_tc", ptr(x_enc), pos_dim, pos_dim, ptr(dirs), ptr(bands), bands.numel(), ptr(sp),
             ptr(cp), Pn, ptr(rgb), ptr(sigma), ctx.pad_value, ptr(_sticky_err(x_enc.device)), stream(),
             work=(Pn * (4.0 * pos_dim + 12 + 16), flops))
        ctx.save_for_backward(x_enc, dirs, bands, sp, cp)
        return rgb, sigma

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g_rgb, g_sigma):
        x_enc, dirs, bands, sp, cp = ctx.saved_tensors
        Pn, pos_dim = x_enc.shape
        g_x = torch.empty_like(x_enc) if ctx.needs_input_grad[0] else None
        g_sp, g_cp = torch.zeros_like(sp), torch.zeros_like(cp)
        work = torch.empty(1, device=x_enc.device, dtype=torch.int32)        # |g|-max of the gradient pre-pass
        flops = 6.0 * Pn * (64 * pos_dim + 16 * 64 + 64 * 43 + 64 * 64 + 3 * 64)
        call("b2n_instant_mlp_bwd_tc", ptr(x_enc), pos_dim, pos_dim, ptr(dirs), ptr(bands), bands.numel(), ptr(sp),
             ptr(cp), Pn, ptr(_c(g_rgb)), ptr(_c(g_sigma)), ptr(g_x), pos_dim, ptr(g_sp), ptr(g_cp), ptr(work),
             ctx.pad_value, ptr(_sticky_err(x_enc.device)), stream(),
             work=(Pn * (8.0 * pos_dim + 12 + 16), flops))
        return g_x, None, None, g_sp, g_cp, None


@torch.no_grad()
def instant_sigma(x_enc, sigma_params, pad_value: float = 0.0):
    """sigma [P,1] of the fused Instant decoder alone: b2n_instant_mlp_fwd_tc with the colour network switched off (no view
    directions, no colour layers).  Same sigma_net arithmetic as ``instant_mlp`` -- bit-identical sigma -- at ~40 % of its
    time; no gradient (occupancy sweeps: DensityGrid.update, SURVEY 8f-3)."""
    require_cuda(x_enc, sigma_params)
    x_enc, sp = _c(x_enc), _c(sigma_params)
    Pn, pos_dim = x_enc.shape
    sigma = _narrow_out(Pn, 1, device=x_enc.device)
    work = (Pn * (4.0 * pos_dim + 4), 2.0 * Pn * (64 * pos_dim + 16 * 64))
    call("b2n_instant_mlp_fwd_tc", ptr(x_enc), pos_dim, pos_dim, None, None, 0, ptr(sp), None, Pn, None, ptr(sigma),
         float(pad_value), ptr(_sticky_err(x_enc.device)), stream(), work=work)
    return sigma


def instant_mlp(x_enc, dirs, bands, sigma_params, color_params, pad_value: float = 0.0):
    """Fused InstantNeRFDecoder on raw unit view directions: (rgb [P,3], sigma [P,1]).  ``pad_value``: content of the
    padded input columns of the two networks (0, or 1 for upstream-tcnn checkpoints: b2n.checkpoint)."""
    return _InstantMLP.apply(x_enc, dirs, bands, sigma_params, color_params, pad_value)


# ----------------------------------------------------------------------------
# 256-wide vanilla NeRF decoder on tcgen05 (bf16 operands, fp32 accumulate in TMEM)
# ----------------------------------------------------------------------------

# The tcgen05 kernels never hang: a stalled mbarrier wait aborts the CTA and raises a device-side flag instead.  Reading
# the flag costs a host sync, so it is checked with a delay -- every 64th launch looks at the flags of earlier launches
# (long finished) -- and a non-zero flag raises here rather than letting garbage activations train on.
_ERR_FLAGS: dict = {}          # device index -> flags of launches not yet inspected
_STICKY_ERR: dict = {}         # device index -> one flag shared by every tcgen05 Instant-decoder launch on that device
_GRAPH_FLAGS: list = []        # abort flags of launches captured into CUDA graphs (state of the latest replay) ...
_GRAPH_OWNERS = __import__("weakref").WeakSet()      # ... or owned by a b2n.graphs.GraphedStep (`_err_flags`), which frees them with itself


def _raise_if_set(flags):
    bad = int(torch.stack(flags).max().item())
    if bad != 0:
        raise RuntimeError(f"a tcgen05 decoder kernel aborted a stalled pipeline (code {bad}); its outputs are invalid")


def _track_err(err: torch.Tensor):
    if torch.cuda.is_current_stream_capturing():
        # inside a CUDA graph (b2n.graphs): no host reads now.  The flag lives in the graph's memory pool, is re-zeroed and
        # re-written by every replay, and is inspected by check_errors() like the sticky flags
        _GRAPH_FLAGS.append(err)
        return
    lst = _ERR_FLAGS.setdefault(err.device.index, [])
    lst.append(err)
    if len(lst) >= 64:
        old = lst[:32]
        del lst[:32]
        _raise_if_set(old)


def _sticky_err(device) -> torch.Tensor:
    """the abort flag of the fused Instant decoder (b2n_instant_mlp_fwd_tc): one int per device, never reset by the
    kernels, read only by ``check_errors`` -- no per-call allocation, memset or host sync, and a stable address for CUDA
    graphs"""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    t = _STICKY_ERR.get(idx)
    if t is None:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("the Instant decoder's abort flag must exist before CUDA-graph capture: run one eager "
                               "step first (b2n.graphs.GraphedStep does)")
        t = _STICKY_ERR[idx] = torch.zeros(1, device=torch.device("cuda", idx), dtype=torch.int32)
    return t


def check_errors():
    """Inspect the abort flags of EVERY tcgen05 launch not looked at yet (one host sync per device).  The delayed check
    above never sees the last < 64 launches of a run; call this where a sync happens anyway -- after ``loss.item()``,
    at the end of ``render_image`` / ``DensityGrid.update`` (done there), after CUDA-graph replays -- so that a short
    evaluation cannot write images computed from an aborted pipeline."""
    for dev in list(_ERR_FLAGS):
        flags, _ERR_FLAGS[dev] = _ERR_FLAGS[dev], []
        if flags:
            _raise_if_set(flags)
    graph_flags = list(_GRAPH_FLAGS)
    for owner in list(_GRAPH_OWNERS):
        graph_flags += owner._err_flags
    by_dev: dict = {}
    for t in graph_flags:
        by_dev.setdefault(t.device.index, []).append(t)
    for flags in by_dev.values():
        _raise_if_set(flags)
    for t in _STICKY_ERR.values():
        if int(t.item()) != 0:
            code = int(t.item())
            t.zero_()
            raise RuntimeError(f"a tcgen05 Instant-decoder kernel aborted a stalled pipeline (code {code}); its outputs "
                               f"are invalid")


def nerf_mlp_supported(decoder, pos_dim: int, dir_dim: int) -> bool:
    """the tcgen05 kernel covers the reference architecture: 8 x 256, skip at 4, view 128"""
    try:
        return (len(decoder.pts_layers) == 8 and decoder.skip_layer == 4 and decoder.feature_layer.out_features == 256
                and decoder.view_layer.out_features == 128 and decoder.pts_layers[0].out_features == 256
                and 0 < pos_dim <= 96 and 0 < dir_dim <= 32)
    except AttributeError:
        return False


def _nerf_mlp_pack(decoder):
    dev = decoder.feature_layer.weight.device
    pos_dim = decoder.pts_layers[0].in_features
    dir_dim = decoder.view_layer.in_features - 256
    ws = [_c(l.weight) for l in decoder.pts_layers]
    ptrs = (ctypes.c_void_p * 8)(*[w.data_ptr() for w in ws])
    fw, vw = _c(decoder.feature_layer.weight), _c(decoder.view_layer.weight)
    packed = torch.empty(_lib.lib.b2n_nerf_mlp_packed_bytes(), device=dev, dtype=torch.uint8)
    call("b2n_nerf_mlp_pack", ptrs, ptr(fw), ptr(vw), pos_dim, dir_dim, ptr(packed), stream())
    bias = torch.cat([l.bias for l in decoder.pts_layers] + [decoder.feature_layer.bias, decoder.view_layer.bias]).float()
    head_bias = torch.cat([decoder.sigma_layer.bias, decoder.rgb_layer.bias]).float()
    return packed, bias.contiguous(), head_bias.contiguous(), pos_dim, dir_dim


@torch.no_grad()
def nerf_mlp_forward(decoder, x_enc, d_enc, save: bool = False):
    """NeRFDecoder forward on the tensor cores.  Returns (rgb [P,3], sigma [P,1], saved planes | None)."""
    require_cuda(x_enc, d_enc)
    if current_rows() is not None:
        raise RuntimeError("the 256-wide tcgen05 decoder does not support a device-side row count (march(static=True))")
    x_enc, d_enc = _c(x_enc), _c(d_enc)
    packed, bias, head_bias, pos_dim, dir_dim = _nerf_mlp_pack(decoder)
    Pn = x_enc.shape[0]
    dev = x_enc.device
    rgb = torch.empty(Pn, 3, device=dev)
    sigma = torch.empty(Pn, 1, device=dev)
    planes = torch.empty(10, Pn, 256, device=dev, dtype=torch.bfloat16) if save else None
    masks = torch.empty(10, Pn, 8, device=dev, dtype=torch.int32) if save else None      # ReLU bits of the planes
    err = torch.zeros(1, device=dev, dtype=torch.int32)
    w_sigma = _c(decoder.sigma_layer.weight).view(-1)
    w_rgb = _c(decoder.rgb_layer.weight).view(-1)
    flops = 2.0 * Pn * (256 * pos_dim + 256 * 256 * 6 + 256 * (256 + pos_dim) + 256 + 256 * 256 + 128 * (256 + dir_dim) + 384)
    call("b2n_nerf_mlp_fwd", ptr(x_enc), pos_dim, ptr(d_enc), dir_dim, ptr(packed), ptr(bias), ptr(w_sigma), ptr(w_rgb),
         ptr(head_bias), Pn, ptr(rgb), ptr(sigma), ptr(planes), ptr(masks), ptr(err), stream(),
         work=(Pn * (4.0 * (pos_dim + dir_dim) + 16 + (5120 if save else 0)), flops))
    _track_err(err)
    return rgb, sigma, (planes, masks) if save else None, err


def _mm_f32(a_t, b):
    """a_t^T @ b for bf16 operands with an fp32 result (plain library GEMM: the weight-gradient
    reductions over all points)."""
    try:
        return torch.mm(a_t.t(), b, out_dtype=torch.float32)
    except TypeError:
        return torch.mm(a_t.t(), b).float()


class _NerfMLP(torch.autograd.Function):
    """NeRFDecoder on tcgen05: forward kernel (saving bf16 layer outputs), backward = the tcgen05
    data-gradient chain + one GEMM per layer for the weight gradients."""

    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, decoder, grad_on, x_enc, d_enc, *params):
        # grad_on: torch.is_grad_enabled() of the CALLER (inside Function.forward grad mode is always off, and
        # needs_input_grad stays True for parameters under torch.no_grad()).  Every evaluation loop of run.py runs under
        # no_grad: nothing is saved there -- the planes are 5 KB per point, 195 GB for one 800 x 800 frame
        need_grad = grad_on and any(ctx.needs_input_grad)
        rgb, sigma, saved, err = nerf_mlp_forward(decoder, x_enc, d_enc, save=need_grad)
        planes, masks = saved if saved is not None else (None, None)
        ctx.decoder = decoder
        ctx.save_for_backward(_c(x_enc), _c(d_enc), rgb, sigma, planes, masks, err)
        return rgb, sigma

    @staticmethod
    @custom_bwd(device_type="cuda")
    def backward(ctx, g_rgb, g_sigma):
        x_enc, d_enc, rgb, sigma, planes, masks, err = ctx.saved_tensors
        dec = ctx.decoder
        if ctx.needs_input_grad[3]:
            raise RuntimeError("tcgen05 NeRFDecoder path does not produce view-direction gradients (use fp32 mode)")
        Pn = x_enc.shape[0]
        dev = x_enc.device
        pos_dim, dir_dim = x_enc.shape[1], d_enc.shape[1]
        ws = [_c(l.weight) for l in dec.pts_layers]
        ptrs = (ctypes.c_void_p * 8)(*[w.data_ptr() for w in ws])
        fw, vw = _c(dec.feature_layer.weight), _c(dec.view_layer.weight)
        packed = torch.empty(_lib.lib.b2n_nerf_mlp_packed_bwd_bytes(), device=dev, dtype=torch.uint8)
        call("b2n_nerf_mlp_pack_bwd", ptrs, ptr(fw), ptr(vw), pos_dim, dir_dim, ptr(packed), stream())
        dz = torch.empty(10, Pn, 256, device=dev, dtype=torch.bfloat16)
        dz_small = torch.empty(Pn, 4, device=dev)
        w_sigma = _c(dec.sigma_layer.weight).view(-1)
        w_rgb = _c(dec.rgb_layer.weight).view(-1)
        flops = 2.0 * Pn * (128 * 256 + 256 * 256 * 8)
        call("b2n_nerf_mlp_bwd", ptr(packed), ptr(w_sigma), ptr(w_rgb), ptr(masks), ptr(rgb), ptr(sigma.view(-1)),
             ptr(_c(g_rgb)), ptr(_c(g_sigma).view(-1)), Pn, ptr(dz), ptr(dz_small), ptr(err), stream(),
             work=(Pn * (2.0 * 5120 + 48), flops))
        # ---- weight / bias gradients: dW = dZ^T In over all points
        # layer inputs in bf16; x / d zero-padded to 64-column multiples (the operand blocks of the tcgen05 kernel)
        kx = 64 if pos_dim <= 64 else 128
        xb = torch.empty(Pn, kx, device=dev, dtype=torch.bfloat16)
        db = torch.empty(Pn, 64, device=dev, dtype=torch.bfloat16)
        call("b2n_pad_bf16", ptr(x_enc), Pn, pos_dim, kx, ptr(xb), stream())
        call("b2n_pad_bf16", ptr(d_enc), Pn, dir_dim, 64, ptr(db), stream())
        H = planes                      # H[0..7] trunk outputs, H[8] feat, H[9][:, :128] hv
        dZ = {l: dz[9 - l] for l in range(8)}     # dZ_l of trunk layer l
        grads = {}
        if Pn >= 64:
            # every layer's weight gradient (but the two 1- / 3-row heads) and all bias column sums: ONE tcgen05 launch
            sizes = [8 * 65536, 256 * kx, 256 * kx, 128 * 256, 128 * 64, 10 * 256]
            flat = torch.zeros(sum(sizes), device=dev)
            dW, dW0, dW4x, dWv_h, dWv_d, gb_all = [t.view(*shape) for t, shape in zip(
                torch.split(flat, sizes), [(8, 256, 256), (256, kx), (256, kx), (128, 256), (128, 64), (10, 256)])]
            call("b2n_nerf_mlp_wgrad", ptr(dz), ptr(planes), ptr(xb), kx, ptr(db), Pn, ptr(dW), ptr(dW0), ptr(dW4x),
                 ptr(dWv_h), ptr(dWv_d), ptr(gb_all), ptr(err), stream(),
                 work=(Pn * (8 * 1024.0 + 2 * (512 + 2 * kx) + 256 + 512 + 128),
                       2.0 * Pn * (8 * 65536 + 2 * 256 * kx + 128 * 256 + 128 * 64)))
            for l in range(8):
                if l == 0:
                    gW = dW0[:, :pos_dim]
                elif l == 4:
                    gW = torch.cat([dW[3], dW4x[:, :pos_dim]], dim=1)
                else:
                    gW = dW[l - 1]
                grads[f"pts{l}"] = (gW, gb_all[9 - l])
            grads["feat"] = (dW[7], gb_all[1])
            grads["view"] = (torch.cat([dWv_h, dWv_d[:, :dir_dim]], dim=1), gb_all[0][:128])
        else:
            gb_all = torch.sum(dz, dim=1, dtype=torch.float32)   # [10, 256] column sums
            for l in range(8):
                if l == 0:
                    gW = _mm_f32(dZ[0], xb)[:, :pos_dim]
                elif l == 4:
                    gW = torch.cat([_mm_f32(dZ[4], H[3]), _mm_f32(dZ[4], xb)[:, :pos_dim]], dim=1)
                else:
                    gW = _mm_f32(dZ[l], H[l - 1])
                grads[f"pts{l}"] = (gW, gb_all[9 - l])
            grads["feat"] = (_mm_f32(dz[1], H[7]), gb_all[1])
            gv = _mm_f32(dz[0], torch.cat([H[8], db], dim=1))[:128]       # [256(128 used), 256 + 64]
            grads["view"] = (gv[:, :256 + dir_dim], gb_all[0][:128])
        # the two small heads (1 x 256 on H_7, 3 x 128 on hv) and their biases: one streaming kernel over the two planes
        heads = torch.zeros(256 + 3 * 128 + 4, device=dev)
        call("b2n_nerf_mlp_head_wgrad", ptr(dz_small), ptr(H[7]), ptr(H[9]), Pn, ptr(heads), heads.data_ptr() + 256 * 4,
             heads.data_ptr() + (256 + 384) * 4, stream(), work=(Pn * (16.0 + 512 + 256), 2.0 * Pn * (256 + 384)))
        small_sum = heads[640:644]
        grads["sigma"] = (heads[:256].view(1, 256), small_sum[3:4])
        grads["rgb"] = (heads[256:640].view(3, 128), small_sum[:3])
        out = []
        for l in range(8):
            out += list(grads[f"pts{l}"])
        for k in ("sigma", "feat", "view", "rgb"):
            out += list(grads[k])
        g_x = None
        if ctx.needs_input_grad[2]:       # d x_enc = dZ0 W0 + dZ4 W4[:, 256:]
            g_x = torch.empty_like(x_enc)
            call("b2n_nerf_mlp_dx", ptr(dz[9]), ptr(dz[5]), ptr(ws[0]), ws[0].stride(0), ws[4].data_ptr() + 256 * 4,
                 ws[4].stride(0), pos_dim, Pn, ptr(g_x), pos_dim, stream(),
                 work=(Pn * (1024.0 + 4.0 * pos_dim), 2.0 * Pn * 512 * pos_dim))
        return (None, None, g_x, None) + tuple(out)


def _nerf_params(decoder):
    ps = []
    for l in decoder.pts_layers:
        ps += [l.weight, l.bias]
    for m in (decoder.sigma_layer, decoder.feature_layer, decoder.view_layer, decoder.rgb_layer):
        ps += [m.weight, m.bias]
    return ps


def nerf_mlp(decoder, x_enc, d_enc):
    """(rgb [P,3], sigma [P,1]) of NeRFDecoder on the tensor cores, differentiable w.r.t. its parameters."""
    if d_enc.requires_grad:
        raise RuntimeError("nerf_mlp: view-direction gradients are not produced by the tcgen05 path")
    return _NerfMLP.apply(decoder, torch.is_grad_enabled(), x_enc, d_enc, *_nerf_params(decoder))


# ----------------------------------------------------------------------------
# fused small-width MLPs of the dynamic configs (bf16 tensor cores): b2n_fmlp_*
# ----------------------------------------------------------------------------

def fused_mlp_supported(d_in: int, hidden: int, n_hidden: int, out_dim: int) -> bool:
    return hidden in (64, 128) and 1 <= n_hidden <= 3 and 1 <= d_in <= 96 and 1 <= out_dim <= 64


class _FusedMLP(torch.autograd.Function):
    """act_out(W_n relu(... relu(W_0 [x0|x1] + b_0) ...) + b_n): forward kernel (saving the bf16 input rows and
    hidden activations when a gradient is needed), backward = the data-gradient chain kernel + one plain GEMM per
    layer for the weight gradients and a column sum per bias."""

    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, x0, x1, out_act, n_layers, grad_on, *wb):
        Ws, bs = list(wb[:n_layers]), list(wb[n_layers:])
        require_cuda(x0, x1, *Ws)
        ctx.rows = current_rows()
        x0, x1 = _c(x0), _c(x1)
        Ws = [W if (W.dtype == torch.float32 and W.stride(-1) == 1) else _c(W) for W in Ws]
        bs = [_c(b) for b in bs]
        Pn, d0 = x0.shape
        d1 = x1.shape[1] if x1 is not None else 0
        hidden, n_hidden, out_dim = Ws[0].shape[0], n_layers - 1, Ws[-1].shape[0]
        dev = x0.device
        need = grad_on and any(ctx.needs_input_grad)      # grad_on: the caller's grad mode (no planes under torch.no_grad())
        in_pad = _lib.lib.b2n_fmlp_in_pad(d0 + d1)
        y = _narrow_out(Pn, out_dim, device=dev) if out_dim <= 4 else torch.empty(Pn, out_dim, device=dev)
        xin = torch.empty(Pn, in_pad, device=dev, dtype=torch.float16) if need else None
        hpl = torch.empty(n_hidden, Pn, hidden, device=dev, dtype=torch.float16) if need else None
        Wp = (ctypes.c_void_p * n_layers)(*[W.data_ptr() for W in Ws])
        ld = (ctypes.c_int * n_layers)(*[W.stride(0) for W in Ws])
        bp = (ctypes.c_void_p * n_layers)(*[(b.data_ptr() if b is not None else None) for b in bs])
        macs = hidden * (d0 + d1) + hidden * hidden * (n_hidden - 1) + out_dim * hidden
        call("b2n_fmlp_fwd", ptr(x0), x0.stride(0), d0, ptr(x1), x1.stride(0) if x1 is not None else 0, d1, hidden,
             n_hidden, Wp, ld, bp, out_dim, out_act, Pn, ptr(y), out_dim, ptr(xin), ptr(hpl), stream(),
             work=(Pn * (4.0 * (d0 + d1 + out_dim) + (2.0 * (in_pad + n_hidden * hidden) if need else 0.0)), 2.0 * Pn * macs))
        ctx.save_for_backward(y, xin, hpl, *Ws)
        ctx.meta = (d0, d1, hidden, n_hidden, out_dim, out_act, n_layers, [b is not None for b in bs])
        return y

    @staticmethod
    @custom_bwd(device_type="cuda")
    @with_ctx_rows
    def backward(ctx, g_y):
        y, xin, hpl, *Ws = ctx.saved_tensors
        d0, d1, hidden, n_hidden, out_dim, out_act, n_layers, has_b = ctx.meta
        Pn = y.shape[0]
        dev = y.device
        g_y = _c(g_y)
        out_pad = _lib.lib.b2n_fmlp_out_pad(out_dim)
        # planes hold S * dZ (see b2n_fmlp_bwd); dz_out is column-summed over ALL allocated rows below, and with a
        # device-side row count the rows behind it are never written: zero-filled (32 bytes per row)
        dz_out = torch.zeros(Pn, out_pad, device=dev, dtype=torch.float16)
        dz_h = torch.empty(n_hidden, Pn, hidden, device=dev, dtype=torch.float16)
        work = torch.empty(2, device=dev, dtype=torch.float32)                    # [0] |g|-max bits, [1] S
        scale = work[1:]
        g_x0 = torch.empty(Pn, d0, device=dev) if ctx.needs_input_grad[0] else None
        g_x1 = torch.empty(Pn, d1, device=dev) if (d1 and ctx.needs_input_grad[1]) else None
        Wp = (ctypes.c_void_p * n_layers)(*[W.data_ptr() for W in Ws])
        ld = (ctypes.c_int * n_layers)(*[W.stride(0) for W in Ws])
        macs = hidden * hidden * (n_hidden - 1) + out_dim * hidden + (hidden * (d0 + d1) if (g_x0 is not None or g_x1 is not None) else 0)
        call("b2n_fmlp_bwd", d0, d1, hidden, n_hidden, Wp, ld, out_dim, out_act, Pn, ptr(y), out_dim, ptr(g_y), out_dim,
             ptr(hpl), ptr(dz_out), ptr(dz_h), ptr(g_x0), d0, ptr(g_x1), d1, ptr(work), stream(),
             work=(Pn * (4.0 * out_dim + 4.0 * n_hidden * hidden + 2.0 * out_pad + 4.0 * (d0 + d1)), 2.0 * Pn * macs))
        shapes = [(Ws[l].shape[0], Ws[l].shape[1]) for l in range(n_layers)]
        in_pad = xin.shape[1]
        if hidden == 128 and Pn >= 64:
            # ---- hidden width 128 (DeformationNetwork): tcgen05 plane GEMMs, TMA-fed, HBM-bound (b2n_fmlp_wgrad_tc)
            sizes = [128 * 128, max(n_hidden - 1, 1) * 128 * 128, 128 * 64, n_hidden * 128]
            flat = torch.zeros(sum(sizes) + 1, device=dev)
            dW0, dWh, dWoT, db_h = [t.view(*shape) for t, shape in zip(
                torch.split(flat[:-1], sizes), [(128, 128), (max(n_hidden - 1, 1), 128, 128), (128, 64), (n_hidden, 128)])]
            err = flat[-1:].view(torch.int32)
            call("b2n_fmlp_wgrad_tc", ptr(dz_h), ptr(dz_out), ptr(hpl), ptr(xin), Pn, n_hidden, in_pad, out_pad, ptr(dW0),
                 ptr(dWh), ptr(dWoT), ptr(db_h), ptr(err), ptr(scale), stream(),
                 work=(2.0 * Pn * ((2 * n_hidden) * 128 + in_pad + out_pad), 2.0 * Pn * (128 * in_pad + (n_hidden - 1) * 16384 + 128 * out_pad)))
            gW = [dW0[:, : shapes[0][1]]] + [dWh[l - 1] for l in range(1, n_hidden)] + [dWoT[:, : shapes[-1][0]].t()]
            gb = [db_h[l] for l in range(n_hidden)] + [torch.sum(dz_out, dim=0, dtype=torch.float32)[: shapes[-1][0]] / scale]
        else:
            # ---- weight / bias gradients of every layer: one launch (b2n_fmlp_wgrad, mma.sync), fp32 accumulation
            n_w = sum(r * c for r, c in shapes)
            flat = torch.zeros(n_w + sum(r for r, _ in shapes), device=dev)
            gW, gb, off, boff = [], [], 0, n_w
            for r, c in shapes:
                gW.append(flat[off:off + r * c].view(r, c))
                gb.append(flat[boff:boff + r])
                off, boff = off + r * c, boff + r
            dzs = [dz_h[l] for l in range(n_hidden)] + [dz_out]
            ins = [xin] + [hpl[l] for l in range(n_hidden)]
            arr_p, arr_i = ctypes.c_void_p * n_layers, ctypes.c_int * n_layers
            call("b2n_fmlp_wgrad", n_layers, arr_p(*[t.data_ptr() for t in dzs]), arr_i(*[t.stride(0) for t in dzs]),
                 arr_i(*[t.shape[1] for t in dzs]), arr_p(*[t.data_ptr() for t in ins]), arr_i(*[t.stride(0) for t in ins]),
                 arr_i(*[t.shape[1] for t in ins]), arr_p(*[g.data_ptr() for g in gW]), arr_i(*[c for _, c in shapes]),
                 arr_i(*[r for r, _ in shapes]), arr_i(*[min(c, t.shape[1]) for (_, c), t in zip(shapes, ins)]),
                 arr_p(*[(gb[l].data_ptr() if has_b[l] else None) for l in range(n_layers)]), Pn, ptr(scale), stream(),
                 work=(2.0 * Pn * sum(a_.shape[1] + b_.shape[1] for a_, b_ in zip(dzs, ins)),
                       2.0 * Pn * sum(r * c for r, c in shapes)))
        gW = [g if ctx.needs_input_grad[5 + l] else None for l, g in enumerate(gW)]
        gb = [gb[l] if (has_b[l] and ctx.needs_input_grad[5 + n_layers + l]) else None for l in range(n_layers)]
        return (g_x0, g_x1, None, None, None) + tuple(gW) + tuple(gb)


def fused_mlp(x0, x1, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]], out_act: str = "none"):
    """Fused ReLU MLP on [x0 | x1] (x1 may be None).  weights[l]: [out, in(+padding columns)] fp32, last = output layer
    (its first out rows are used -- pass ``W[:out_dim]`` for a padded FullyFusedMLP matrix); biases[l] or None."""
    n = len(weights)
    hidden = weights[0].shape[0]
    d_in = x0.shape[1] + (x1.shape[1] if x1 is not None else 0)
    if not fused_mlp_supported(d_in, hidden, n - 1, weights[-1].shape[0]):
        raise ValueError("fused_mlp: unsupported shape (hidden 64/128, 1..3 hidden layers, <= 96 inputs, <= 64 outputs)")
    return _FusedMLP.apply(x0, x1, _ACT[out_act], n, torch.is_grad_enabled(), *weights, *biases)
