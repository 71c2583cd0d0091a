"""Fast inference rendering: march only the occupied samples, in waves, and stop each ray once its transmittance falls
below ``t_min`` (b2n_render_* of include/b2nerf.h; the contract is documented there and in DESIGN.md §5g).

    out = render_image_fast(model, rays_o, rays_d, near, far, 128, density_grid=grid)    # [H,W,3] rays
    out.color, out.depth, out.acc, out.n_evaluated, out.n_waves

This is not the reference's ``render_rays``: with ``t_min = 0`` it equals ``render_rays(..., perturb=False,
density_grid=grid)`` up to the order of the transmittance product; with ``t_min > 0`` colour and acc are within
``t_min`` of that, depth within ``t_min * far``.  Each wave hands the next K active samples of every ray still alive to
the model in one call, so a wave's buffers stay near ``WAVE_POINTS`` samples whatever the image size.  Every wave reads
two 4-byte counts on the host, so a render cannot be captured into a CUDA graph.

``render_rays_train`` is the training render itself (march -> model -> composite), the body that
``src/renderer.py::render_rays`` and ``b2n.render_rays_distortion`` share.
"""
from __future__ import annotations

from typing import NamedTuple

import numpy as np
import torch

from . import march as _march
from ._lib import active_rows, call, lib, ptr, require_cuda, stream
from .ops import check_errors, composite, distortion

MAX_SAMPLES = 1024
WAVE_POINTS = 2 ** 21          # samples per model call, at most: the fastest in `tools/kbench.py render` (DESIGN.md §5g)


class Rendered(NamedTuple):
    color: torch.Tensor        # [B,3] (render_image_fast: [H,W,3])
    depth: torch.Tensor        # [B]   ([H,W])
    acc: torch.Tensor          # [B]   ([H,W])
    n_evaluated: int           # samples the model was called on
    n_waves: int


def samples_per_wave(n_alive: int, n_samples: int) -> int:
    """K = clamp(pow2_floor(WAVE_POINTS / n_alive), 1, N): few samples per ray while many rays are alive (most of them
    stop at the first opaque surface), more as rays finish."""
    k = max(1, WAVE_POINTS // max(n_alive, 1))
    return min(1 << (k.bit_length() - 1), n_samples)


def _check_rays(rays_o, rays_d, n_samples, t_min):
    if not isinstance(rays_o, torch.Tensor) or not isinstance(rays_d, torch.Tensor):
        raise ValueError("rays_o and rays_d must be torch tensors")
    if rays_o.dim() != 2 or rays_o.shape[-1] != 3 or rays_d.shape != rays_o.shape:
        raise ValueError(f"rays_o and rays_d must both be [B,3], got {tuple(rays_o.shape)} and {tuple(rays_d.shape)}")
    if isinstance(n_samples, bool) or not isinstance(n_samples, (int, np.integer)):
        raise ValueError(f"n_samples must be an int, got {n_samples!r}")
    if not 1 <= int(n_samples) <= MAX_SAMPLES:
        raise ValueError(f"n_samples must be in [1, {MAX_SAMPLES}], got {n_samples}")
    t_min = float(t_min)
    if not (0.0 <= t_min < 1.0):                   # NaN fails too
        raise ValueError(f"t_min must be finite with 0 <= t_min < 1, got {t_min}")
    return int(n_samples), t_min


def render_rays_train(model, rays_o, rays_d, near, far, n_samples, perturb, density_grid=None, times=None,
                      white_bkgd=True, bg_color=None, _jitter=None, with_distortion=False):
    """The body of the training render (src/renderer.py::render_rays, and b2n.render_rays_distortion with
    ``with_distortion``): march -> model -> composite, plus the per-ray distortion of the same samples when asked.
    Returns (color, depth, acc, extras, dist): ``extras`` is the dict render_rays returns for a dynamic model given
    ``times`` (else None), ``dist`` [B] the distortion (else None)."""
    device = rays_o.device
    n_rays = rays_o.shape[0]
    mode = getattr(model, "mode", "unknown")
    dynamic = mode in ("part3", "part4")
    if bg_color is None:
        bg_color = torch.ones(3, device=device) if white_bkgd else torch.zeros(3, device=device)
    ray_times = None
    if dynamic:
        ray_times = times if times is not None else torch.zeros((n_rays, 1), device=device)
        if ray_times.shape != (n_rays, 1):
            raise ValueError("times must have shape [n_rays, 1]")
    u = None
    if perturb:
        u = _jitter if _jitter is not None else torch.rand((n_rays, n_samples), device=device)

    if density_grid is not None:
        m = _march.march(rays_o, rays_d, near, far, n_samples, u, bits=density_grid.bits(),
                         R=density_grid.resolution, bound=density_grid.bound, times=ray_times)
    else:
        m = _march.march(rays_o, rays_d, near, far, n_samples, u, times=ray_times)

    # static mode (b2n.march.set_static_capacity): the number of valid rows of the compact buffers lives on the device
    dist = None
    with active_rows(m.n_dev):
        if dynamic:
            rgb, sigma, delta_x = model(m.pts, m.dirs, t=m.times)
        else:
            rgb, sigma = model(m.pts, m.dirs)
            delta_x = None
        want_dx = times is not None and dynamic and delta_x is not None
        sigma = sigma.float()
        color, depth, acc, mean_dx = composite(rgb.float(), sigma, m.z, rays_d, bg=bg_color,
                                               dx=delta_x.float() if want_dx else None,
                                               mask_words=m.mask_words, ray_offset=m.ray_offset)
        if with_distortion:
            dist = distortion(sigma, m.z, rays_d, near, far, mask_words=m.mask_words, ray_offset=m.ray_offset)
    if times is None:
        return color, depth, acc, None, dist
    extras = {}
    if want_dx:
        extras["mean_delta_x"] = mean_dx
    return color, depth, acc, extras, dist


@torch.no_grad()
def render_rays_fast(model, rays_o, rays_d, near, far, n_samples, density_grid=None, times=None, white_bkgd=True,
                     bg_color=None, t_min=1e-4, _samples_per_wave=None) -> Rendered:
    """Render rays ``rays_o``, ``rays_d`` [B,3] with the samples of ``render_rays(..., perturb=False,
    density_grid=density_grid)``: depths ``b2n.march.z_tables(near, far, n_samples)`` (no jitter), and only the
    samples whose voxel is set in ``density_grid`` (all of them without a grid).  A ray stops after the first sample
    that leaves its transmittance below ``t_min`` (0 <= t_min < 1; 0 never stops a ray).

    The model is called as ``render_rays`` calls it -- ``model(pts, dirs)``, or ``model(pts, dirs, t=...)`` with the
    ray's time for the dynamic models (Part 3 / Part 4; ``times`` [B,1], zeros when None) -- under ``no_grad`` in eval
    mode; its previous mode is restored afterwards.  ``bg_color``: [3] or [B,3]; when None, white (``white_bkgd``) or
    black.  ``_samples_per_wave`` (private, tests only) forces K.  Returns ``Rendered(color [B,3], depth [B], acc [B],
    n_evaluated, n_waves)``."""
    N, eps = _check_rays(rays_o, rays_d, n_samples, t_min)
    require_cuda(rays_o, rays_d, times, bg_color)
    dev = rays_o.device
    B = rays_o.shape[0]
    dynamic = getattr(model, "mode", "unknown") in ("part3", "part4")
    if bg_color is None:
        bg_color = torch.ones(3, device=dev) if white_bkgd else torch.zeros(3, device=dev)
    if bg_color.shape not in ((3,), (B, 3)):
        raise ValueError(f"bg_color must be [3] or [B,3], got {tuple(bg_color.shape)}")
    bg = bg_color.float().contiguous()
    ray_t = None
    if dynamic:
        ray_t = times if times is not None else torch.zeros((B, 1), device=dev)
        if ray_t.shape != (B, 1):
            raise ValueError("times must have shape [n_rays, 1]")
        ray_t = ray_t.float().contiguous()
    if _samples_per_wave is not None and not 1 <= int(_samples_per_wave):
        raise ValueError("_samples_per_wave must be >= 1")
    color = torch.empty(B, 3, device=dev)
    depth = torch.empty(B, device=dev)
    acc = torch.empty(B, device=dev)
    if B == 0:
        return Rendered(color, depth, acc, 0, 0)
    rays_o, rays_d = rays_o.float().contiguous(), rays_d.float().contiguous()

    zb = _march.z_tables(near, far, N, dev)[0]
    W = (N + 31) // 32
    words = torch.empty(B, W, device=dev, dtype=torch.int32)
    counts = torch.empty(B, device=dev, dtype=torch.int32)
    bits, R, bound = (None, 0, 1.0) if density_grid is None else \
        (density_grid.bits(), int(density_grid.resolution), float(density_grid.bound))
    scale = float(np.float32(R / (2 * bound))) if bits is not None else 0.0
    call("b2n_march_mask", ptr(rays_o), ptr(rays_d), ptr(zb), None, None, None, ptr(bits), R, bound, scale, B, N, None,
         ptr(words), ptr(counts), stream())
    if bits is not None:                           # only for the forced sample of an all-empty mask (render_rays does it)
        offs = torch.empty(B + 1, device=dev, dtype=torch.int32)
        total = torch.empty(1, device=dev, dtype=torch.int32)
        scan_scratch = torch.empty(lib.b2n_march_scan_scratch(B), device=dev, dtype=torch.uint8)
        call("b2n_march_scan", ptr(counts), ptr(words), W, B, ptr(offs), ptr(total), ptr(scan_scratch), stream())
        del offs, total, scan_scratch

    state = torch.empty(B, 8, device=dev, dtype=torch.int32)               # 32 bytes per ray, layout owned by the library
    alive, alive_next = (torch.empty(B, device=dev, dtype=torch.int32) for _ in range(2))
    scratch = torch.empty(int(lib.b2n_render_scratch(B)), device=dev, dtype=torch.uint8)
    dev_counts = torch.empty(2, device=dev, dtype=torch.int32)           # [0]: alive rays, [1]: samples of the wave
    call("b2n_render_begin", ptr(words), B, N, ptr(state), ptr(alive), ptr(dev_counts[0:1]), ptr(scratch), stream())
    n_alive = int(dev_counts[0].item())
    n_evaluated = n_waves = 0
    was_training = model.training
    model.eval()
    try:
        while n_alive > 0:
            K = min(int(_samples_per_wave), N) if _samples_per_wave is not None else samples_per_wave(n_alive, N)
            cap = n_alive * K
            sidx = torch.empty(cap, device=dev, dtype=torch.int32)
            pts = torch.empty(cap, 3, device=dev)
            dirs = torch.empty(cap, 3, device=dev)
            t_out = torch.empty(cap, 1, device=dev) if dynamic else None
            call("b2n_render_emit", ptr(rays_o), ptr(rays_d), ptr(ray_t), ptr(zb), ptr(words), B, N, ptr(state),
                 ptr(alive), n_alive, K, ptr(sidx), ptr(pts), ptr(dirs), ptr(t_out), ptr(dev_counts[1:2]),
                 ptr(scratch), stream())
            P = int(dev_counts[1].item())
            if dynamic:
                rgb, sigma, _ = model(pts[:P], dirs[:P], t=t_out[:P])
            else:
                rgb, sigma = model(pts[:P], dirs[:P])
            rgb = rgb.float().reshape(-1, 3).contiguous()
            sigma = sigma.float().reshape(-1).contiguous()
            call("b2n_render_composite", ptr(rgb), ptr(sigma), ptr(zb), ptr(rays_d), B, N, eps, ptr(state),
                 ptr(alive), n_alive, ptr(sidx), ptr(alive_next), ptr(dev_counts[0:1]), ptr(scratch), stream())
            alive, alive_next = alive_next, alive
            n_evaluated += P
            n_waves += 1
            n_alive = int(dev_counts[0].item())
    finally:
        model.train(was_training)
    call("b2n_render_finish", ptr(state), B, ptr(bg), int(bg.dim() == 2), ptr(color), ptr(depth), ptr(acc), stream())
    check_errors()                                 # the outputs are about to be read: no silent garbage
    return Rendered(color, depth, acc, n_evaluated, n_waves)


def render_image_fast(model, rays_o, rays_d, near, far, n_samples, density_grid=None, times=None, white_bkgd=True,
                      bg_color=None, t_min=1e-4, _samples_per_wave=None) -> Rendered:
    """``render_rays_fast`` over the rays of an image, ``rays_o`` / ``rays_d`` [H,W,3] (``times`` [H,W,1] or [H*W,1],
    ``bg_color`` [3] or [H,W,3]): colour [H,W,3], depth and acc [H,W].  No ``chunk`` argument: the wave buffers are
    bounded by the per-wave sample budget, not by the image size."""
    if not isinstance(rays_o, torch.Tensor) or rays_o.dim() != 3 or rays_o.shape[-1] != 3:
        raise ValueError(f"rays_o must be [H,W,3], got {getattr(rays_o, 'shape', rays_o)}")
    if not isinstance(rays_d, torch.Tensor) or rays_d.shape != rays_o.shape:
        raise ValueError(f"rays_d must be [H,W,3] like rays_o, got {getattr(rays_d, 'shape', rays_d)}")
    h, w = rays_o.shape[:2]
    if times is not None:
        times = times.reshape(-1, 1)
    if bg_color is not None and bg_color.dim() == 3:
        bg_color = bg_color.reshape(-1, 3)
    out = render_rays_fast(model, rays_o.reshape(-1, 3), rays_d.reshape(-1, 3), near, far, n_samples,
                           density_grid=density_grid, times=times, white_bkgd=white_bkgd, bg_color=bg_color,
                           t_min=t_min, _samples_per_wave=_samples_per_wave)
    return Rendered(out.color.view(h, w, 3), out.depth.view(h, w), out.acc.view(h, w), out.n_evaluated, out.n_waves)
