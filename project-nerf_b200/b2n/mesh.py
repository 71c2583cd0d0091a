"""Triangle-mesh export of a trained field: a sigma sweep over a full-resolution lattice and marching-tetrahedra surface
extraction on the GPU (b2n_mesh_* of include/b2nerf.h; the extraction rules are documented there and in DESIGN.md §5f).

    sigma = density_lattice(model, 512, bound)          # [R,R,R] on the model's device, x slowest
    verts, faces = extract(sigma, threshold, bound)     # closed, consistently wound mesh of sigma > threshold
    write_ply("field.ply", verts, faces)

``extract_mesh(model, resolution, threshold, bound, t=None)`` runs the first two in turn.
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import call, lib, ptr, require_cuda, stream

MAX_RESOLUTION = 1024
SWEEP_BATCH = 2 ** 21          # points per model call: DensityGrid.update's batch


def lattice_axis(resolution: int, bound: float, device) -> torch.Tensor:
    """The 1-D axis of the lattice: ``torch.linspace(-bound, bound, resolution)`` on ``device`` (fp32), exactly as
    ``DensityGrid`` builds it (the values are torch's, not ``-bound + i*h``)."""
    return torch.linspace(-bound, bound, resolution, device=device, dtype=torch.float32)


def _check_resolution(resolution):
    if isinstance(resolution, bool) or not isinstance(resolution, (int, np.integer)):
        raise ValueError(f"resolution must be an int, got {resolution!r}")
    if not 2 <= int(resolution) <= MAX_RESOLUTION:
        raise ValueError(f"resolution must be in [2, {MAX_RESOLUTION}], got {resolution}")
    return int(resolution)


def _check_bound(bound):
    bound = float(bound)
    if not (bound > 0.0 and np.isfinite(bound)):
        raise ValueError(f"bound must be finite and > 0, got {bound}")
    return bound


@torch.no_grad()
def density_lattice(model, resolution: int, bound: float, t=None) -> torch.Tensor:
    """sigma [R,R,R] (fp32, on the model's device) of ``model`` on the lattice ``axis x axis x axis``,
    ``axis = linspace(-bound, bound, R)``, index [ix,iy,iz] with x slowest -- the lattice of ``DensityGrid``.

    The sweep calls ``model.density(x[, t])`` on batches of 2^21 points built on the device from the 1-D axis (the
    R^3 x 3 point array is never materialised); a model without ``density`` is called like ``DensityGrid.update``
    calls it, with zero view directions.  ``t``: scalar time for the dynamic models (Part 3 / Part 4).  The model runs
    in eval mode (train mode perturbs the coordinates) and gets its previous mode back afterwards."""
    R = _check_resolution(resolution)
    bound = _check_bound(bound)
    params = next(iter(model.parameters()), None)
    device = params.device if params is not None else torch.device("cuda")
    ax = lattice_axis(R, bound, device)
    n = R ** 3
    out = torch.empty(n, device=device, dtype=torch.float32)
    density = getattr(model, "density", None)
    was_training = model.training
    model.eval()
    try:
        for i in range(0, n, SWEEP_BATCH):
            j = min(i + SWEEP_BATCH, n)
            idx = torch.arange(i, j, device=device)
            x = torch.stack((ax[idx // (R * R)], ax[(idx // R) % R], ax[idx % R]), dim=-1)
            tt = None if t is None else torch.full((j - i, 1), float(t), device=device, dtype=torch.float32)
            if density is not None:
                s = density(x) if tt is None else density(x, t=tt)
            elif tt is None:
                _, s = model(x, torch.zeros_like(x))
            else:
                _, s, _ = model(x, torch.zeros_like(x), t=tt)
            out[i:j] = s.reshape(-1)
    finally:
        model.train(was_training)
    return out.view(R, R, R)


def extract(sigma: torch.Tensor, threshold: float, bound: float):
    """(verts [V,3] fp32, faces [F,3] int32) of the closed surface sigma = threshold of a lattice already on the GPU.

    ``sigma`` [R,R,R] fp32 contiguous CUDA tensor over ``linspace(-bound, bound, R)`` per axis (x slowest), 2 <= R <= 1024;
    a point is inside when sigma > threshold (threshold > 0).  The lattice is padded with a ring where sigma = 0, so the
    mesh is closed even where the region touches the box.  Faces share vertices by index and are wound so that normals
    point outwards; two calls give bitwise-equal output.  One host synchronisation (the two totals).  A mesh with 2^31 or
    more vertices or faces is refused."""
    if not isinstance(sigma, torch.Tensor):
        raise ValueError("sigma must be a torch tensor")
    require_cuda(sigma)
    if sigma.dtype != torch.float32:
        raise ValueError(f"sigma must be float32, got {sigma.dtype}")
    if sigma.dim() != 3 or not (sigma.shape[0] == sigma.shape[1] == sigma.shape[2]):
        raise ValueError(f"sigma must be a cubic [R,R,R] lattice, got shape {tuple(sigma.shape)}")
    if not sigma.is_contiguous():
        raise ValueError("sigma must be contiguous")
    R = _check_resolution(sigma.shape[0])
    tau = float(threshold)
    if not (tau > 0.0 and np.isfinite(np.float32(tau))):
        raise ValueError(f"threshold must be finite and > 0, got {threshold}")
    bound = _check_bound(bound)
    dev = sigma.device
    ax = lattice_axis(R, bound, dev)
    h = ax[1:2] - ax[0:1]
    ext = torch.cat([ax[:1] - h, ax, ax[-1:] + h]).contiguous()
    scratch = torch.empty(int(lib.b2n_mesh_scratch(R)), device=dev, dtype=torch.uint8)
    totals = torch.empty(2, device=dev, dtype=torch.int64)
    call("b2n_mesh_count", ptr(sigma), R, tau, ptr(scratch), ptr(totals), stream())
    V, F = (int(v) for v in totals.cpu())
    if V >= 2 ** 31 or F >= 2 ** 31:
        raise ValueError(f"mesh too large: {V} vertices and {F} faces, int32 face indices address fewer than 2^31 "
                         "(lower the resolution)")
    verts = torch.empty(V, 3, device=dev, dtype=torch.float32)
    faces = torch.empty(F, 3, device=dev, dtype=torch.int32)
    if V > 0:
        call("b2n_mesh_emit", ptr(sigma), ptr(ext), R, tau, ptr(scratch), V, F, ptr(verts), ptr(faces), stream())
    return verts, faces


def extract_mesh(model, resolution: int, threshold: float, bound: float, t=None):
    """``extract(density_lattice(model, resolution, bound, t), threshold, bound)``"""
    return extract(density_lattice(model, resolution, bound, t), threshold, bound)


def write_ply(path, verts, faces) -> None:
    """Binary little-endian PLY: float x, y, z per vertex, a uchar-counted int list of 3 vertex ids per face."""
    v = np.ascontiguousarray(torch.as_tensor(verts).detach().cpu().numpy(), dtype="<f4").reshape(-1, 3)
    f = np.ascontiguousarray(torch.as_tensor(faces).detach().cpu().numpy(), dtype="<i4").reshape(-1, 3)
    rec = np.empty(len(f), dtype=[("n", "u1"), ("v", "<i4", (3,))])
    rec["n"] = 3
    rec["v"] = f
    header = ("ply\nformat binary_little_endian 1.0\n"
              f"element vertex {len(v)}\nproperty float x\nproperty float y\nproperty float z\n"
              f"element face {len(f)}\nproperty list uchar int vertex_indices\nend_header\n")
    with open(path, "wb") as fh:
        fh.write(header.encode("ascii"))
        fh.write(v.tobytes())
        fh.write(rec.tobytes())
