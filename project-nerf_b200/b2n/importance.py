"""Hierarchical importance sampling: resample every ray from the weights of a coarse pass and composite the coarse and
fine samples together (b2n_importance_sample of include/b2nerf.h; the contract is documented there and in DESIGN.md §5h).

    out = render_rays_hierarchical(model, rays_o, rays_d, near, far, 64, 128, perturb=True)
    out.color, out.depth, out.acc                    # the fine render over the 64 + 128 merged samples
    out.coarse_color, out.coarse_depth, out.coarse_acc

This is NeRF's hierarchical sampling (Mildenhall et al. 2020) with one shared network: the coarse pass is exactly
``render_rays(..., n_coarse, perturb)``; the fine depths come from the coarse weights (no gradient flows through them,
as in NeRF); the model is then called on the fine points only, and its coarse outputs are reused in the fine composite
instead of being evaluated a second time.  The reference has no such pass, so ``render_rays`` / ``render_image`` are
unchanged and this is a separate entry point.
"""
from __future__ import annotations

from typing import Dict, NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import march as _march
from .ops import check_errors, composite
from ._lib import call, ptr, require_cuda, stream

MAX_SAMPLES = 1024             # n_coarse + n_fine: the compositing limit

_U_TABLES: Dict[Tuple[int, str], torch.Tensor] = {}


class Hierarchical(NamedTuple):
    color: torch.Tensor                   # [B,3] fine render (render_image_hierarchical: [H,W,3])
    depth: torch.Tensor                   # [B]
    acc: torch.Tensor                     # [B]
    coarse_color: torch.Tensor            # [B,3] the coarse pass, = render_rays(..., n_coarse, perturb)
    coarse_depth: torch.Tensor            # [B]
    coarse_acc: torch.Tensor              # [B]
    z: torch.Tensor                       # [B, n_coarse + n_fine] merged depths, non-decreasing
    mean_delta_x: Optional[torch.Tensor]  # [B,3] of the fine render: dynamic models with ``times`` only


def u_table(n_fine: int, device) -> torch.Tensor:
    """the deterministic fine positions torch.linspace(0, 1, n_fine), built once per (n_fine, device)"""
    key = (int(n_fine), str(device))
    hit = _U_TABLES.get(key)
    if hit is None:
        hit = _U_TABLES[key] = torch.linspace(0.0, 1.0, steps=int(n_fine), device=device).contiguous()
    return hit


def _check_counts(n_coarse, n_fine):
    for name, v in (("n_coarse", n_coarse), ("n_fine", n_fine)):
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"{name} must be an int, got {v!r}")
    n_coarse, n_fine = int(n_coarse), int(n_fine)
    if n_coarse < 3 or n_fine < 1 or n_coarse + n_fine > MAX_SAMPLES:
        raise ValueError(f"need n_coarse >= 3, n_fine >= 1 and n_coarse + n_fine <= {MAX_SAMPLES}, "
                         f"got {n_coarse} + {n_fine}")
    return n_coarse, n_fine


def importance_sample(sigma, z, rays_d, n_fine, u_jitter=None):
    """The fine depths of NeRF's sample_pdf and their merge with the coarse ones (b2n_importance_sample).
    sigma, z [B,Nc] fp32 (z sorted per ray), rays_d [B,3]; ``u_jitter`` [B,n_fine] U[0,1) for stratified fine
    positions, None for torch.linspace(0, 1, n_fine).  Returns (z_fine [B,n_fine], z_merged [B,Nc+n_fine],
    merge_src [B,Nc+n_fine] int32).  No gradient."""
    require_cuda(sigma, z, rays_d, u_jitter)
    B, Nc = z.shape
    Nc, Nf = _check_counts(Nc, n_fine)
    if sigma.shape != (B, Nc) or rays_d.shape != (B, 3):
        raise ValueError(f"need sigma [B,Nc] and rays_d [B,3] with z [B,Nc] = {tuple(z.shape)}, "
                         f"got {tuple(sigma.shape)} and {tuple(rays_d.shape)}")
    if u_jitter is not None and u_jitter.shape != (B, Nf):
        raise ValueError(f"u_jitter must be [B, n_fine] = {(B, Nf)}, got {tuple(u_jitter.shape)}")
    dev = z.device
    sigma, z, rays_d = (t.detach().float().contiguous() for t in (sigma, z, rays_d))
    table = None if u_jitter is not None else u_table(Nf, dev)
    if u_jitter is not None:
        u_jitter = u_jitter.detach().float().contiguous()
    z_fine = torch.empty(B, Nf, device=dev)
    z_merged = torch.empty(B, Nc + Nf, device=dev)
    merge_src = torch.empty(B, Nc + Nf, device=dev, dtype=torch.int32)
    call("b2n_importance_sample", ptr(sigma), ptr(z), ptr(rays_d), ptr(table), ptr(u_jitter), B, Nc, Nf,
         ptr(z_fine), ptr(z_merged), ptr(merge_src), stream(),
         work=(B * (8.0 * Nc + 12.0 + (4.0 * Nf if u_jitter is not None else 0.0) + 4.0 * Nf + 8.0 * (Nc + Nf)), 0.0))
    return z_fine, z_merged, merge_src


def _gather(coarse, fine, index):
    """per-sample values [B*Nc, C] and [B*Nf, C] in merged order [B*(Nc+Nf), C] (differentiable)"""
    B, M = index.shape
    both = torch.cat([coarse.reshape(B, -1, coarse.shape[-1]), fine.reshape(B, -1, fine.shape[-1])], dim=1)
    return torch.gather(both, 1, index.unsqueeze(-1).expand(B, M, both.shape[-1])).reshape(B * M, -1)


def render_rays_hierarchical(model, rays_o, rays_d, near, far, n_coarse, n_fine, perturb, times=None,
                             white_bkgd=True, bg_color=None, _jitter=None, _jitter_fine=None) -> Hierarchical:
    """Render rays ``rays_o``, ``rays_d`` [B,3] with ``n_coarse`` stratified samples in [near, far] and ``n_fine``
    samples drawn from the coarse weights (b2n_importance_sample), composited together over the merged depths.

    The model is called as ``render_rays`` calls it -- ``model(pts, dirs)``, or ``model(pts, dirs, t=...)`` for the
    dynamic models (Part 3 / Part 4; ``times`` [B,1], zeros when None) -- once on the B * n_coarse coarse points and
    once on the B * n_fine fine points.  ``perturb``: jittered coarse strata and stratified fine positions; otherwise
    the unperturbed depths and torch.linspace(0, 1, n_fine).  ``bg_color``: [3] or [B,3]; when None, white
    (``white_bkgd``) or black.  Gradients reach the model through both composites; the fine depths carry none.
    ``_jitter`` [B,n_coarse] / ``_jitter_fine`` [B,n_fine] (private, tests only) replace the torch.rand draws."""
    Nc, Nf = _check_counts(n_coarse, n_fine)
    if not isinstance(rays_o, torch.Tensor) or not isinstance(rays_d, torch.Tensor) or rays_o.dim() != 2 \
            or rays_o.shape[-1] != 3 or rays_d.shape != rays_o.shape:
        raise ValueError(f"rays_o and rays_d must both be [B,3], got {getattr(rays_o, 'shape', rays_o)} and "
                         f"{getattr(rays_d, 'shape', rays_d)}")
    require_cuda(rays_o, rays_d, times, bg_color, _jitter, _jitter_fine)
    dev = rays_o.device
    B = rays_o.shape[0]
    dynamic = getattr(model, "mode", "unknown") in ("part3", "part4")
    if bg_color is None:
        bg_color = torch.ones(3, device=dev) if white_bkgd else torch.zeros(3, device=dev)
    ray_t = None
    if dynamic:
        ray_t = times if times is not None else torch.zeros((B, 1), device=dev)
        if ray_t.shape != (B, 1):
            raise ValueError("times must have shape [n_rays, 1]")
    for name, j, n in (("_jitter", _jitter, Nc), ("_jitter_fine", _jitter_fine, Nf)):
        if j is not None and j.shape != (B, n):
            raise ValueError(f"{name} must be [B, {n}], got {tuple(j.shape)}")
    u = u_f = None
    if perturb:
        u = _jitter if _jitter is not None else torch.rand((B, Nc), device=dev)
        u_f = _jitter_fine if _jitter_fine is not None else torch.rand((B, Nf), device=dev)

    def field(pts, dirs, t):
        if dynamic:
            rgb, sigma, dx = model(pts, dirs, t=t)
        else:
            (rgb, sigma), dx = model(pts, dirs), None
        return rgb.float().reshape(-1, 3), sigma.float().reshape(-1), (None if dx is None else dx.float().reshape(-1, 3))

    # 1. the coarse pass: render_rays(..., n_coarse, perturb) without an occupancy grid
    m = _march.march(rays_o, rays_d, near, far, Nc, u, times=ray_t)
    rgb_c, sig_c, dx_c = field(m.pts, m.dirs, m.times)
    cc, cd, ca, _ = composite(rgb_c, sig_c, m.z, rays_d, bg=bg_color)
    # 2. fine depths from the coarse weights (no gradient) and their merge with the coarse depths
    z_fine, z_merged, merge_src = importance_sample(sig_c.view(B, Nc), m.z, rays_d, Nf, u_f)
    # 3. the model on the fine points only
    ro, rd = rays_o.float().contiguous(), rays_d.float().contiguous()
    t_in = None if ray_t is None else ray_t.float().contiguous()
    Pf = B * Nf
    pts, dirs = torch.empty(Pf, 3, device=dev), torch.empty(Pf, 3, device=dev)
    t_f = torch.empty(Pf, 1, device=dev) if t_in is not None else None
    call("b2n_march_compact", ptr(ro), ptr(rd), ptr(t_in), ptr(z_fine), None, None, B, Nf, None, ptr(pts), ptr(dirs),
         ptr(t_f), stream(), work=(Pf * (4.0 + 24.0 + (4.0 if t_f is not None else 0.0)) + B * 24.0, 0.0))
    rgb_f, sig_f, dx_f = field(pts, dirs, t_f)
    # 4. the coarse outputs are reused: every sample of the fine composite comes from one of the two model calls
    idx = merge_src.long()
    rgb = _gather(rgb_c, rgb_f, idx)
    sigma = _gather(sig_c.unsqueeze(-1), sig_f.unsqueeze(-1), idx).reshape(-1)
    want_dx = times is not None and dynamic and dx_f is not None
    dx = _gather(dx_c, dx_f, idx) if want_dx else None
    # 5. the fine composite over the merged depths
    color, depth, acc, mdx = composite(rgb, sigma, z_merged, rays_d, bg=bg_color, dx=dx)
    return Hierarchical(color, depth, acc, cc, cd, ca, z_merged, mdx if want_dx else None)


@torch.no_grad()
def render_image_hierarchical(model, rays_o, rays_d, near, far, n_coarse, n_fine, chunk, white_bkgd) -> Hierarchical:
    """``render_rays_hierarchical(..., perturb=False)`` over the rays of an image, ``rays_o`` / ``rays_d`` [H,W,3], in
    chunks of ``chunk`` rays, in eval mode (the model's previous mode is restored afterwards, also when it raises).
    Colours [H,W,3], depths and acc [H,W], merged depths [H,W,n_coarse+n_fine]."""
    if not isinstance(rays_o, torch.Tensor) or rays_o.dim() != 3 or rays_o.shape[-1] != 3:
        raise ValueError(f"rays_o must be [H,W,3], got {getattr(rays_o, 'shape', rays_o)}")
    if not isinstance(rays_d, torch.Tensor) or rays_d.shape != rays_o.shape:
        raise ValueError(f"rays_d must be [H,W,3] like rays_o, got {getattr(rays_d, 'shape', rays_d)}")
    Nc, Nf = _check_counts(n_coarse, n_fine)
    if isinstance(chunk, bool) or not isinstance(chunk, (int, np.integer)) or chunk < 1:
        raise ValueError(f"chunk must be a positive int, got {chunk!r}")
    h, w = rays_o.shape[:2]
    ro, rd = rays_o.reshape(-1, 3), rays_d.reshape(-1, 3)
    was_training = model.training
    model.eval()
    try:
        parts = [render_rays_hierarchical(model, ro[i:i + chunk], rd[i:i + chunk], near, far, Nc, Nf, False,
                                          white_bkgd=white_bkgd)
                 for i in range(0, ro.shape[0], int(chunk))]
    finally:
        model.train(was_training)
    check_errors()                                 # the image is about to be read by the caller: no silent garbage
    cat = [torch.cat([p[i] for p in parts]) for i in range(7)]
    return Hierarchical(cat[0].view(h, w, 3), cat[1].view(h, w), cat[2].view(h, w), cat[3].view(h, w, 3),
                        cat[4].view(h, w), cat[5].view(h, w), cat[6].view(h, w, Nc + Nf), None)
