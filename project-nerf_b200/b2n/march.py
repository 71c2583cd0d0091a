"""Host side of the ray-marching front end (sampling, occupancy, compaction).

Replaces src/renderer.py:186-201 (sample_stratified), :134-166
(get_active_mask) and the boolean-mask gathers of :290-323 of the reference
with the b2n_march_* / b2n_occ_* kernels.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import numpy as np
import torch

from ._lib import call, lib, ptr, require_cuda, stream

_Z_TABLES: Dict[Tuple, Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = {}


def z_tables(near: float, far: float, n_samples: int, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(z_base, z_lo, z_hi), each [N]: the unperturbed depths and stratum bounds of
    src/renderer.py:189-197, built ONCE per (near, far, N, device) with the very
    torch ops the reference uses, so the kernel's z = lo + (hi - lo) * u is
    bit-identical to the reference's."""
    key = (float(near), float(far), int(n_samples), str(device))
    hit = _Z_TABLES.get(key)
    if hit is not None:
        return hit
    t = torch.linspace(0.0, 1.0, steps=n_samples, device=device)
    z = near * (1.0 - t) + far * t
    mids = 0.5 * (z[1:] + z[:-1])
    hi = torch.cat([mids, z[-1:]])
    lo = torch.cat([z[:1], mids])
    out = (z.contiguous(), lo.contiguous(), hi.contiguous())
    _Z_TABLES[key] = out
    return out


def pack_occupancy(binary_grid: torch.Tensor) -> torch.Tensor:
    """torch.bool [R,R,R] -> uint32 bitfield (viewed as int32) of ceil(R^3/32) words."""
    require_cuda(binary_grid)
    b = binary_grid.contiguous()
    n = b.numel()
    bits = torch.empty((n + 31) // 32, device=b.device, dtype=torch.int32)
    call("b2n_occ_pack_bits", ptr(b.view(torch.uint8)), n, ptr(bits), stream())
    return bits


def active_mask(pts: torch.Tensor, bits: torch.Tensor, R: int, bound: float) -> torch.Tensor:
    """DensityGrid.get_active_mask (src/renderer.py:134-166) on the bitfield."""
    require_cuda(pts, bits)
    pts = pts.float().contiguous()
    Pn = pts.shape[0]
    mask = torch.empty(Pn, device=pts.device, dtype=torch.bool)
    scale = float(np.float32(R / (2 * bound)))
    call("b2n_occ_active_mask", ptr(pts), Pn, ptr(bits), R, float(bound), scale, ptr(mask.view(torch.uint8)), stream())
    return mask


class Marched:
    """Result of marching a ray batch: depths, activity bitmask, compact sample list.  ``n_dev`` (static mode only):
    int32[1] device tensor with the number of valid rows of ``pts`` / ``dirs`` / ``times`` (their first dimension is then
    the fixed capacity B * N, ``n_active`` too)."""
    __slots__ = ("z", "mask_words", "ray_offset", "n_active", "n_dev", "pts", "dirs", "times", "sample_idx", "B", "N")


_STATIC = {"on": False}


def set_static_capacity(on: bool):
    """Static mode: ``march`` behind an occupancy grid never reads the active-sample count on the host.  The compact
    buffers get the fixed capacity B * N and the count stays on the device (``Marched.n_dev``); ``render_rays`` hands it
    to every kernel of the step through ``b2n._lib.active_rows``.  No host synchronisation is left in a training step, so
    it can be captured into a CUDA graph (b2n.graphs.GraphedStep) and the host can run ahead of the device.  Costs
    capacity-sized allocations (and torch glue ops over capacity rows in the dynamic models); needs the 16-bit fused
    decoders.  Default off: the exact-size path with its single 4-byte read per call (the reference syncs three times:
    renderer.py:309-323)."""
    _STATIC["on"] = bool(on)


def static_capacity() -> bool:
    return _STATIC["on"]


def march(rays_o: torch.Tensor, rays_d: torch.Tensor, near: float, far: float, n_samples: int,
          u: Optional[torch.Tensor], bits: Optional[torch.Tensor] = None, R: int = 0, bound: float = 1.0,
          times: Optional[torch.Tensor] = None, want_idx: bool = False) -> Marched:
    """Depths + (optional) occupancy test + ordered compaction of the active samples.

    With ``bits`` the number of active samples is data dependent, so exactly one
    4-byte device->host read sizes the compact buffers (the reference syncs three
    times per call: renderer.py:309,316,332).

    When ``rays_o`` or ``rays_d`` requires grad (and grad mode is on), ``pts`` is differentiable w.r.t. both
    (b2n_march_points_bwd; pose refinement, DESIGN.md §5k) with the same values.  ``dirs``, ``times``, ``z`` and the
    mask never carry a gradient."""
    require_cuda(rays_o, rays_d, u, bits, times)
    rays_o, rays_d = rays_o.float().contiguous(), rays_d.float().contiguous()
    B, N = rays_o.shape[0], int(n_samples)
    dev = rays_o.device
    zb, zlo, zhi = z_tables(near, far, N, dev)
    m = Marched()
    m.B, m.N = B, N
    m.n_dev = None
    W = (N + 31) // 32
    m.z = torch.empty(B, N, device=dev)
    if times is not None:
        times = times.float().contiguous()
    m.sample_idx = None
    if B == 0:
        m.mask_words = m.ray_offset = None
        m.n_active = 0
        m.pts = torch.empty(0, 3, device=dev)
        m.dirs = torch.empty(0, 3, device=dev)
        m.times = torch.empty(0, 1, device=dev) if times is not None else None
        return m
    words = torch.empty(B, W, device=dev, dtype=torch.int32)
    counts = torch.empty(B, device=dev, dtype=torch.int32)
    if u is not None:
        u = u.float().contiguous()
    scale = float(np.float32(R / (2 * bound))) if bits is not None else 0.0
    call("b2n_march_mask", ptr(rays_o), ptr(rays_d), ptr(zb), ptr(zlo), ptr(zhi), ptr(u), ptr(bits), int(R),
         float(bound), scale, B, N, ptr(m.z), ptr(words), ptr(counts), stream(),
         work=(B * (24.0 + 4.0 * N * (2 if u is not None else 1) + 4.0 * W + 4.0), 0.0))      # o, d, U in; z, words, count out
    if bits is None:
        m.mask_words, m.ray_offset, m.n_active = None, None, B * N
    else:
        offs = torch.empty(B + 1, device=dev, dtype=torch.int32)
        total = torch.empty(1, device=dev, dtype=torch.int32)
        scratch = torch.empty(lib.b2n_march_scan_scratch(B), device=dev, dtype=torch.uint8)
        call("b2n_march_scan", ptr(counts), ptr(words), W, B, ptr(offs), ptr(total), ptr(scratch), stream(),
             work=(B * (8.0 + 4.0), 0.0))
        m.mask_words, m.ray_offset = words, offs
        if _STATIC["on"]:
            m.n_active, m.n_dev = B * N, total     # fixed capacity, count stays on the device
        else:
            m.n_active = int(total.item())        # the one host sync of the masked path
    if torch.is_grad_enabled() and (rays_o.requires_grad or rays_d.requires_grad):
        m.pts = _Points.apply(rays_o, rays_d, times, m, want_idx)
    else:
        m.pts = _compact(rays_o, rays_d, times, m, want_idx)
    return m


def _compact(rays_o, rays_d, times, m, want_idx):
    """b2n_march_compact: fills m.dirs, m.times, m.sample_idx (if asked) and returns the points"""
    Pn, B, N, dev = m.n_active, m.B, m.N, rays_o.device
    W = (N + 31) // 32
    pts = torch.empty(Pn, 3, device=dev)
    m.dirs = torch.empty(Pn, 3, device=dev)
    m.times = torch.empty(Pn, 1, device=dev) if times is not None else None
    if want_idx:
        m.sample_idx = torch.empty(Pn, device=dev, dtype=torch.int32)
    call("b2n_march_compact", ptr(rays_o), ptr(rays_d), ptr(times), ptr(m.z), ptr(m.mask_words), ptr(m.ray_offset),
         B, N, ptr(m.sample_idx), ptr(pts), ptr(m.dirs), ptr(m.times), stream(),
         work=(Pn * (4.0 + 24.0 + (4.0 if times is not None else 0.0)) + B * (24.0 + 4.0 * W + 4.0), 0.0))
    return pts


class _Points(torch.autograd.Function):
    """The points o + d * z of ``march`` as a function of the rays (pose refinement, DESIGN.md §5k): the forward is the
    same b2n_march_compact call, the backward b2n_march_points_bwd.  dirs, times, z and the mask stay constants."""

    @staticmethod
    def forward(ctx, rays_o, rays_d, times, m, want_idx):
        pts = _compact(rays_o, rays_d, times, m, want_idx)
        ctx.save_for_backward(m.z, m.mask_words, m.ray_offset)
        ctx.n_active = m.n_active
        return pts

    @staticmethod
    def backward(ctx, g_pts):
        z, words, offs = ctx.saved_tensors
        B, N = z.shape
        g_pts = g_pts.float().contiguous()
        g_o = torch.empty(B, 3, device=g_pts.device)
        g_d = torch.empty(B, 3, device=g_pts.device)
        call("b2n_march_points_bwd", ptr(z), ptr(words), ptr(offs), ptr(g_pts), B, N, ptr(g_o), ptr(g_d), stream(),
             work=(ctx.n_active * 12.0 + B * (4.0 * N + 4.0 * ((N + 31) // 32) + 28.0), 0.0))
        return g_o, g_d, None, None, None
