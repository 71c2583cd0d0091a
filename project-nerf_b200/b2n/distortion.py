"""Training render with the distortion loss of mip-NeRF 360 (Barron et al. 2022, eq. 15; b2n_distortion_* of
include/b2nerf.h, the contract is documented there and in DESIGN.md §5j).

    color, depth, acc, dist = render_rays_distortion(model, rays_o, rays_d, near, far, 128, True, density_grid=grid)
    loss = mse(color, target) + 0.01 * dist.mean()        # mip-NeRF 360 uses lambda = 0.01

The term pulls the weights of every ray together into one compact interval, which removes the semi-transparent
floaters and background haze an occupancy-grid model otherwise learns.  The render is exactly ``render_rays`` (the same
march -> model -> composite; colour, depth and acc are bitwise its outputs) with the per-ray distortion of the same
samples appended; its gradient reaches the model through sigma only.  The reference has no such term, so
``render_rays`` / ``render_image`` are unchanged and this is a separate entry point.
"""
from __future__ import annotations

from .render import render_rays_train


def render_rays_distortion(model, rays_o, rays_d, near, far, n_samples, perturb, density_grid=None, times=None,
                           white_bkgd=True, bg_color=None, _jitter=None):
    """``render_rays`` with the same arguments, plus the distortion [B] of its samples (``b2n.distortion`` over the
    marched depths and the model's sigma, in the compact layout when ``density_grid`` is given): (color, depth, acc,
    dist), or (color, depth, acc, dist, extras) for a dynamic model given ``times`` -- the extras dict stays last."""
    color, depth, acc, extras, dist = render_rays_train(
        model, rays_o, rays_d, near, far, n_samples, perturb, density_grid=density_grid, times=times,
        white_bkgd=white_bkgd, bg_color=bg_color, _jitter=_jitter, with_distortion=True)
    if extras is None:
        return color, depth, acc, dist
    return color, depth, acc, dist, extras
