"""GPU tests of camera pose refinement (b2n.PoseRefinement, b2n_sample_rays_bwd and b2n_march_points_bwd of
include/b2nerf.h): the rays at xi = 0 against sample_random_rays bit for bit and at xi != 0 against the float64 oracle
of _pose_oracle.py, both backward kernels against float64 sums within their rounding bound, determinism and the
layouts of the march, the end-to-end gradient against a torch-glue path over the same model kernels, CUDA-graph capture
of a static-capacity step, and training that recovers perturbed poses on the checker-band sphere."""
import json
import math
import os

import numpy as np
import pytest
import torch

import _pose_oracle as PO
from _util import GOLDEN, record

pytestmark = pytest.mark.gpu
DEV = "cuda"
NEAR, FAR = 2.0, 6.0
U = 2.0 ** -24
INSTANT = dict(mode="part2_instant", scene_bound=1.5, n_levels=8, log2_hashmap_size=14, base_resolution=16,
               per_level_scale=1.5, L_embed_dir=4, hidden_dim=64)
VANILLA = dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)


def _tiny(cls_name="blender", scene_scale=0.5):
    from src.dataset import BlenderDataset, DynamicDataset
    cls = BlenderDataset if cls_name == "blender" else DynamicDataset
    return cls(os.path.join(GOLDEN, "dataset_tiny"), split="train", white_bkgd=True, scene_scale=scene_scale)


def _xi(V, seed, scale=0.05):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(V, 6, generator=g) * scale).to(DEV)


# ---- rays
@pytest.mark.parametrize("tag", ["blender", "dynamic"])
def test_rays_at_zero_are_sample_random_rays_bitwise(tag):
    import b2n
    from b2n import errormap
    ds = _tiny(tag)
    refine = b2n.PoseRefinement(len(ds))
    torch.manual_seed(77)
    ref = ds.sample_random_rays(257, DEV)
    torch.manual_seed(77)
    picks = tuple(t.to(DEV) for t in ds._draw(257, "cpu"))
    out = refine.rays(ds, picks)
    assert len(out) == len(ref) == (4 if tag == "dynamic" else 3)
    for a, b in zip(out, ref):
        assert torch.equal(a, b)
    assert out[0].requires_grad and out[1].requires_grad and not out[2].requires_grad
    emap = b2n.ErrorMap(len(ds), ds.H, ds.W, cells=(6, 5))
    picks, _ = emap.sample(1000, generator=torch.Generator(device=DEV).manual_seed(1))
    for a, b in zip(refine.rays(ds, picks), errormap.rays(ds, picks)):
        assert torch.equal(a, b)
    # a whole view: what get_image_rays builds on the host, to fp32 rounding (its rotation is a matmul)
    ro, rd, tgt = refine.image_rays(ds, 2)[:3]
    hro, hrd, htgt = ds.get_image_rays(2, DEV)[:3]
    assert ro.shape == hro.shape and tgt.shape == htgt.shape
    assert torch.allclose(ro, hro, atol=1e-6, rtol=0) and torch.allclose(rd, hrd, atol=1e-6, rtol=0)
    assert torch.equal(tgt, htgt)


def test_rays_at_nonzero_xi_match_the_oracle():
    import b2n
    ds = _tiny("blender", scene_scale=0.5)
    V = len(ds)
    refine = b2n.PoseRefinement(V)
    xi = _xi(V, 3)
    with torch.no_grad():
        refine.delta.copy_(xi)
    g = torch.Generator().manual_seed(4)
    picks = tuple(torch.randint(0, n, (4096,), generator=g).to(DEV) for n in (V, ds.H, ds.W))
    ro, rd, _ = refine.rays(ds, picks)
    P = PO.corrected(ds.poses, xi.cpu())
    o, d = PO.rays(P, *(t.cpu() for t in picks), ds.H, ds.W, ds.focal, 0.5)
    err_o = float((ro.cpu().double() - o).abs().max() / o.abs().max())
    err_d = float((rd.cpu().double() - d).abs().max())
    record("pose rays vs oracle at xi != 0: max |o - o_ref| / max|o_ref|", err_o)
    record("pose rays vs oracle at xi != 0: max |d - d_ref|", err_d)
    assert err_o < 32 * U and err_d < 32 * U, (err_o, err_d)
    # only the views in the mask move; their corrections get gradient, the others exactly none
    mask = torch.arange(V, device=DEV) % 2 == 0
    part = b2n.PoseRefinement(V, refine=mask)
    with torch.no_grad():
        part.delta.copy_(xi)
    ro2, rd2, _ = part.rays(ds, picks)
    keep = ~mask[picks[0]]
    from b2n import errormap
    ro0, rd0, _ = errormap.rays(ds, picks)
    assert torch.equal(ro2[keep], ro0[keep]) and torch.equal(rd2[keep], rd0[keep])
    (ro2.sum() + rd2.sum()).backward()
    assert torch.equal(part.delta.grad[~mask], torch.zeros_like(part.delta.grad[~mask]))
    assert bool((part.delta.grad[mask].abs().sum(-1) > 0).all())


# ---- b2n_march_points_bwd
def _march_rays(B, seed):
    from b2n import synthetic
    ro, rd, _ = synthetic.random_rays(B, seed=seed)
    return ro.to(DEV), rd.to(DEV)


def _points_bwd(m, g_pts):
    from b2n._lib import call, ptr, stream
    g_o = torch.full((m.B, 3), float("nan"), device=DEV)
    g_d = torch.full((m.B, 3), float("nan"), device=DEV)
    call("b2n_march_points_bwd", ptr(m.z), ptr(m.mask_words), ptr(m.ray_offset), ptr(g_pts.contiguous()), m.B, m.N,
         ptr(g_o), ptr(g_d), stream())
    return g_o, g_d


def _bits(kind, R=64):
    from b2n import march, synthetic
    if kind == "dense":
        return None
    occ = synthetic.ball_occupancy(R, 1.5, 1.0) if kind == "compact" else torch.zeros(R, R, R, dtype=torch.bool)
    return march.pack_occupancy(occ.to(DEV))


def _check_points_bwd(m, g_pts, g_o, g_d, tag):
    B, N = m.B, m.N
    idx = m.sample_idx.long()
    dense = torch.zeros(B * N, 3, dtype=torch.float64, device=DEV)
    dense[idx] = g_pts[:idx.numel()].double()
    dense = dense.view(B, N, 3)
    ref_o, ref_d = PO.points_bwd(m.z, dense)
    cnt = torch.zeros(B * N, dtype=torch.float64, device=DEV)
    cnt[idx] = 1.0
    n_r = cnt.view(B, N).sum(-1, keepdim=True)
    bound_o = (n_r + 1) * U * dense.abs().sum(1) + 1e-30
    bound_d = (n_r + 1) * U * (m.z.double()[..., None] * dense).abs().sum(1) + 1e-30
    r_o = float(((g_o.double() - ref_o).abs() / bound_o).max())
    r_d = float(((g_d.double() - ref_d).abs() / bound_d).max())
    record(f"march_points_bwd vs fp64 sums / (n+1) 2^-24 sum|terms| ({tag})", max(r_o, r_d))
    assert r_o <= 1.0 and r_d <= 1.0, (tag, r_o, r_d)


@pytest.mark.parametrize("layout", ["dense", "compact"])
@pytest.mark.parametrize("N", [1, 65, 128, 1024])
def test_march_points_bwd_matches_fp64_sums(N, layout):
    from b2n import march
    B = 2048 if N < 1024 else 512
    ro, rd = _march_rays(B, seed=N)
    u = torch.rand(B, N, device=DEV, generator=torch.Generator(DEV).manual_seed(N))
    m = march.march(ro, rd, NEAR, FAR, N, u, bits=_bits(layout), R=64, bound=1.5, want_idx=True)
    g_pts = torch.randn(m.n_active, 3, device=DEV, generator=torch.Generator(DEV).manual_seed(N + 1))
    g_o, g_d = _points_bwd(m, g_pts)
    _check_points_bwd(m, g_pts, g_o, g_d, f"N={N} {layout}")
    g_o2, g_d2 = _points_bwd(m, g_pts)
    assert torch.equal(g_o, g_o2) and torch.equal(g_d, g_d2)           # two runs: the same bits
    # through autograd: the same points as without a gradient, and the backward is this kernel
    o_, d_ = ro.clone().requires_grad_(True), rd.clone().requires_grad_(True)
    m2 = march.march(o_, d_, NEAR, FAR, N, u, bits=_bits(layout), R=64, bound=1.5)
    assert m2.pts.requires_grad and not m2.dirs.requires_grad and not m2.z.requires_grad
    assert torch.equal(m2.pts.detach(), m.pts) and torch.equal(m2.dirs, m.dirs) and torch.equal(m2.z, m.z)
    ga, gb = torch.autograd.grad(m2.pts, (o_, d_), g_pts)
    assert torch.equal(ga, g_o) and torch.equal(gb, g_d)
    with torch.no_grad():
        assert not march.march(o_, d_, NEAR, FAR, N, u, bits=_bits(layout), R=64, bound=1.5).pts.requires_grad


def test_march_points_bwd_all_empty_grid():
    from b2n import march
    B, N = 256, 64
    ro, rd = _march_rays(B, seed=5)
    m = march.march(ro, rd, NEAR, FAR, N, None, bits=_bits("empty"), R=64, bound=1.5, want_idx=True)
    assert m.n_active == 1                                                # the forced sample 0 of ray 0
    g_pts = torch.randn(1, 3, device=DEV)
    g_o, g_d = _points_bwd(m, g_pts)
    assert torch.equal(g_o[0], g_pts[0]) and torch.equal(g_d[0], m.z[0, 0] * g_pts[0])
    assert torch.equal(g_o[1:], torch.zeros(B - 1, 3, device=DEV)) and torch.equal(g_d[1:], torch.zeros(B - 1, 3, device=DEV))


def test_march_points_bwd_static_capacity_reads_no_row_behind_the_count():
    from b2n import march
    B, N = 4096, 128
    ro, rd = _march_rays(B, seed=9)
    u = torch.rand(B, N, device=DEV)
    bits = _bits("compact")
    m0 = march.march(ro, rd, NEAR, FAR, N, u, bits=bits, R=64, bound=1.5)
    n = m0.n_active
    g_pts = torch.randn(n, 3, device=DEV)
    ref_o, ref_d = _points_bwd(m0, g_pts)
    try:
        march.set_static_capacity(True)
        m = march.march(ro, rd, NEAR, FAR, N, u, bits=bits, R=64, bound=1.5)
    finally:
        march.set_static_capacity(False)
    assert int(m.n_dev.item()) == n and m.n_active == B * N
    cap = torch.full((B * N, 3), float("nan"), device=DEV)                # garbage behind the device count
    cap[:n] = g_pts
    g_o, g_d = _points_bwd(m, cap)
    assert torch.equal(g_o, ref_o) and torch.equal(g_d, ref_d)


# ---- b2n_sample_rays_bwd
H_S, W_S, F_S, SCALE_S = 64, 48, 52.5, 0.8


def _rays_bwd(poses, picks, g_o, g_d, out=None):
    from b2n._lib import call, lib, ptr, stream
    V, B = poses.shape[0], picks[0].shape[0]
    g = torch.full((V, 4, 4), float("nan"), device=DEV) if out is None else out
    scratch = torch.empty(int(lib.b2n_sample_rays_bwd_scratch(B, V)), dtype=torch.uint8, device=DEV)
    call("b2n_sample_rays_bwd", ptr(poses), *(ptr(t) for t in picks), B, V, H_S, W_S, F_S, SCALE_S, ptr(g_o), ptr(g_d),
         ptr(g), ptr(scratch), stream())
    return g


def _abs_terms(poses, picks, g_o, g_d):
    """per view, sum over its rays of |each term| of g_R and g_t, and the ray count (float64)"""
    img, y, x = (t.cpu() for t in picks)
    V = poses.shape[0]
    c = PO.cam_dirs(y, x, H_S, W_S, F_S)
    M = poses.cpu().double()[img]
    d = (M[:, :3, :3] @ c[..., None])[..., 0]
    n = d.norm(dim=-1, keepdim=True)
    dh = d / n
    gd = g_d.cpu().double()
    gr = (gd - dh * (dh * gd).sum(-1, keepdim=True)) / n
    terms = torch.zeros(img.shape[0], 4, 4, dtype=torch.float64)
    terms[:, :3, :3] = (gr[:, :, None] * c[:, None, :]).abs()
    terms[:, :3, 3] = (SCALE_S * g_o.cpu().double()).abs()
    out = torch.zeros(V, 4, 4, dtype=torch.float64).index_add_(0, img, terms)
    cnt = torch.zeros(V, dtype=torch.float64).index_add_(0, img, torch.ones(img.shape[0], dtype=torch.float64))
    return out, cnt


def _check_rays_bwd(poses, picks, g_o, g_d, got, tag):
    ref = PO.rays_bwd(poses.cpu(), *(t.cpu() for t in picks), H_S, W_S, F_S, SCALE_S, g_o.cpu(), g_d.cpu())
    terms, cnt = _abs_terms(poses, picks, g_o, g_d)
    bound = cnt[:, None, None] * U * terms + 1e-30
    ratio = float(((got.cpu().double() - ref).abs() / bound).max())
    record(f"sample_rays_bwd vs fp64 oracle / n_v 2^-24 sum|terms| ({tag})", ratio)
    assert ratio <= 1.0, (tag, ratio)
    assert torch.equal(got[:, 3, :], torch.zeros_like(got[:, 3, :]))
    empty = cnt == 0
    assert torch.equal(got[empty.to(DEV)], torch.zeros_like(got[empty.to(DEV)]))
    return ref


@pytest.mark.parametrize("V", [1, 100, 1000])
def test_sample_rays_bwd_matches_the_oracle(V):
    from b2n import synthetic
    B = 8192
    poses = synthetic.hemisphere_poses(V, seed=V).to(DEV)
    g = torch.Generator().manual_seed(V)
    img = torch.randint(0, V, (B,), generator=g)
    if V > 1:
        img[img % 5 == 0] = (img[img % 5 == 0] + 1) % V                    # views that receive no rays
        img[img % 5 == 0] = (img[img % 5 == 0] + 1) % V
    picks = (img.to(DEV), torch.randint(0, H_S, (B,), generator=g).to(DEV), torch.randint(0, W_S, (B,), generator=g).to(DEV))
    g_o, g_d = torch.randn(B, 3, generator=g).to(DEV), torch.randn(B, 3, generator=g).to(DEV)
    got = _rays_bwd(poses, picks, g_o, g_d)
    _check_rays_bwd(poses, picks, g_o, g_d, got, f"V={V}")
    assert torch.equal(got, _rays_bwd(poses, picks, g_o, g_d))          # two runs: the same bits
    perm = torch.randperm(B, generator=g).to(DEV)                          # the same rays in another order
    shuffled = _rays_bwd(poses, tuple(t[perm] for t in picks), g_o[perm], g_d[perm])
    _check_rays_bwd(poses, picks, g_o, g_d, shuffled, f"V={V} shuffled")


def test_sample_rays_bwd_one_view_and_out_of_range_ids():
    from b2n import synthetic
    V, B = 100, 2 ** 16
    poses = synthetic.hemisphere_poses(V, seed=3).to(DEV)
    g = torch.Generator().manual_seed(5)
    y, x = torch.randint(0, H_S, (B,), generator=g).to(DEV), torch.randint(0, W_S, (B,), generator=g).to(DEV)
    g_o, g_d = torch.randn(B, 3, generator=g).to(DEV), torch.randn(B, 3, generator=g).to(DEV)
    picks = (torch.full((B,), 37, dtype=torch.int64, device=DEV), y, x)   # every ray in one view
    got = _rays_bwd(poses, picks, g_o, g_d)
    _check_rays_bwd(poses, picks, g_o, g_d, got, "all rays in one view")
    # ids outside [0, V): never summed, nothing written outside g_poses
    img = torch.randint(0, V, (B,), generator=g)
    bad = torch.rand(B, generator=g) < 0.1
    img[bad] = torch.where(torch.rand(B, generator=g) < 0.5, -1, V)[bad]
    buf = torch.full(((V + 2) * 16,), 7.0, device=DEV)
    out = buf[16:16 + 16 * V].view(V, 4, 4)
    _rays_bwd(poses, (img.to(DEV), y, x), g_o, g_d, out=out)
    assert torch.equal(buf[:16], torch.full((16,), 7.0, device=DEV)) and torch.equal(buf[-16:], torch.full((16,), 7.0, device=DEV))
    keep = (~bad).to(DEV)
    _check_rays_bwd(poses, (img.to(DEV)[keep], y[keep], x[keep]), g_o[keep], g_d[keep], out, "out-of-range ids dropped")


# ---- end-to-end gradient
def _model(cfg, seed=0):
    from src.core import NeuralField
    torch.manual_seed(seed)
    return NeuralField(cfg).to(DEV).train()


def _grid():
    from b2n import synthetic
    from src.renderer import DensityGrid
    grid = DensityGrid(resolution=64, bound=1.5).to(DEV)
    grid.binary_grid = synthetic.ball_occupancy(64, 1.5, 1.0).to(DEV)
    return grid


def _glue_grad(model, refine, ds, picks, u, N, grid, G):
    """g_xi by torch ops: rays from corrected_poses, points o[ray] + d[ray] z over march(..., want_idx=True); the ray
    values are the kernel's (the torch rays carry only the gradient), so both paths hand the model the same points"""
    from b2n import march
    from b2n.ops import composite
    ro_k, rd_k, _ = refine.rays(ds, picks)
    ro_k, rd_k = ro_k.detach(), rd_k.detach()
    img, y, x = picks
    poses = ds._resident(torch.device(DEV))[0]
    P = refine.corrected_poses(poses)[img]
    f = float(np.float32(ds.focal))
    c = torch.stack([(x.float() - ds.W * 0.5) / f, -((y.float() - ds.H * 0.5) / f), -torch.ones_like(x, dtype=torch.float32)], -1)
    d = (P[:, :3, :3] * c[:, None, :]).sum(-1)
    d = d / d.norm(dim=-1, keepdim=True)
    o = P[:, :3, 3] * ds.scene_scale
    o_g, d_g = ro_k + (o - o.detach()), rd_k + (d - d.detach())
    kw = dict(bits=grid.bits(), R=grid.resolution, bound=grid.bound) if grid is not None else {}
    m = march.march(ro_k, rd_k, NEAR, FAR, N, u, want_idx=True, **kw)
    idx = m.sample_idx.long()
    r = idx // N
    pts = o_g[r] + d_g[r] * m.z.reshape(-1)[idx][:, None]
    rgb, sigma = model(pts, m.dirs)
    color, depth, _, _ = composite(rgb.float(), sigma.float(), m.z, rd_k, bg=torch.ones(3, device=DEV),
                                   mask_words=m.mask_words, ray_offset=m.ray_offset)
    loss = (color * G[:, :3]).sum() + (depth * G[:, 3]).sum()
    return torch.autograd.grad(loss, refine.delta)[0]


def _new_grad(model, refine, ds, picks, u, N, grid, G):
    from src.renderer import render_rays
    ro, rd, _ = refine.rays(ds, picks)
    color, depth, _ = render_rays(model, ro, rd, NEAR, FAR, N, True, density_grid=grid,
                                  bg_color=torch.ones(3, device=DEV), _jitter=u)
    loss = (color * G[:, :3]).sum() + (depth * G[:, 3]).sum()
    return torch.autograd.grad(loss, refine.delta)[0]


@pytest.mark.parametrize("grid_on", [False, True], ids=["no_grid", "grid"])
@pytest.mark.parametrize("case", ["instant_fp32", "instant_bf16", "nerf_fp32", "nerf_bf16"])
def test_end_to_end_gradient_matches_torch_glue(case, grid_on):
    import b2n
    ds = _tiny("blender", scene_scale=1.0)
    V, B, N = len(ds), 512, 64
    cfg = INSTANT if case.startswith("instant") else VANILLA
    prev = b2n.mlp_precision()
    b2n.set_mlp_precision(case.split("_")[1])
    try:
        model = _model(cfg)
        refine = b2n.PoseRefinement(V)
        with torch.no_grad():
            refine.delta.copy_(_xi(V, 11, scale=0.01))
        g = torch.Generator().manual_seed(12)
        picks = tuple(torch.randint(0, n, (B,), generator=g).to(DEV) for n in (V, ds.H, ds.W))
        u = torch.rand(B, N, generator=g).to(DEV)
        G = torch.randn(B, 4, generator=g).to(DEV)
        grid = _grid() if grid_on else None
        new = _new_grad(model, refine, ds, picks, u, N, grid, G)
        glue = _glue_grad(model, refine, ds, picks, u, N, grid, G)
    finally:
        b2n.set_mlp_precision(prev)
    assert torch.isfinite(new).all() and float(glue.abs().max()) > 0
    err = float((new - glue).abs().max() / glue.abs().max())
    record(f"pose end-to-end g_xi vs torch glue, max|diff|/max|g| ({case}, grid={grid_on})", err)
    assert err < 1e-4, (case, grid_on, err)


def test_static_capacity_step_graph_replay_equals_eager():
    import b2n
    from b2n import march
    from src.renderer import render_rays
    ds = _tiny("blender", scene_scale=1.0)
    V, B, N = len(ds), 1024, 64
    prev = b2n.mlp_precision()
    b2n.set_mlp_precision("bf16")
    march.set_static_capacity(True)
    try:
        model = _model(INSTANT)
        refine = b2n.PoseRefinement(V)
        with torch.no_grad():
            refine.delta.copy_(_xi(V, 21, scale=0.01))
        g = torch.Generator().manual_seed(22)
        picks = tuple(torch.randint(0, n, (B,), generator=g).to(DEV) for n in (V, ds.H, ds.W))
        u = torch.rand(B, N, generator=g).to(DEV)
        G = torch.randn(B, 3, generator=g).to(DEV)
        grid = _grid()
        grid.bits()

        def step():
            ro, rd, _ = refine.rays(ds, picks)
            color = render_rays(model, ro, rd, NEAR, FAR, N, True, density_grid=grid,
                                bg_color=torch.ones(3, device=DEV), _jitter=u)[0]
            return torch.autograd.grad((color * G).sum(), refine.delta)[0]

        eager = step()
        assert torch.equal(eager, step())                                 # deterministic
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = step()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
        b2n.check_errors()
    finally:
        march.set_static_capacity(False)
        b2n.set_mlp_precision(prev)


# ---- training recovers perturbed poses
SCENE_CFG = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
                 per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
RADIUS, BAND = 0.6, 0.25


def _band_scene(ro, rd):
    """the checker-band sphere of test_gpu_errormap.py: white background, a shaded sphere, a black-and-white checker
    of 24 x 6 squares on the band |n_z| < BAND (its colour breaks the sphere's symmetry)"""
    b = (ro * rd).sum(-1)
    disc = b * b - ((ro * ro).sum(-1) - RADIUS ** 2)
    hit = disc > 0
    n = (ro + rd * (-b - torch.sqrt(disc.clamp_min(0)))[:, None]) / RADIUS
    col = torch.stack([0.5 + 0.5 * n[:, 2], 0.2 + 0.0 * n[:, 0], 0.5 - 0.5 * n[:, 2]], -1)
    band = hit & (n[:, 2].abs() < BAND)
    az = torch.atan2(n[:, 1], n[:, 0])
    check = ((torch.floor(az * 24 / (2 * np.pi)) + torch.floor(n[:, 2] * 6 / (2 * BAND))) % 2)[:, None].expand(-1, 3)
    col = torch.where(band[:, None], check, col)
    return torch.where(hit[:, None], col, torch.ones_like(col))


def _write_dataset(root, true_poses, stored_poses, H):
    from PIL import Image
    from b2n import synthetic
    os.makedirs(os.path.join(root, "train"), exist_ok=True)
    frames = []
    for i, (pt, ps) in enumerate(zip(true_poses, stored_poses)):
        ro, rd = synthetic.image_rays(pt, H=H, W=H)
        col = _band_scene(ro.double(), rd.double()).reshape(H, H, 3)
        rgba = np.concatenate([(col.numpy() * 255).round().astype(np.uint8), np.full((H, H, 1), 255, np.uint8)], -1)
        Image.fromarray(rgba, "RGBA").save(os.path.join(root, "train", f"r_{i}.png"))
        frames.append({"file_path": f"./train/r_{i}", "transform_matrix": ps.tolist()})
    with open(os.path.join(root, "transforms_train.json"), "w") as f:
        json.dump({"camera_angle_x": synthetic.CAMERA_ANGLE_X, "frames": frames}, f)


def _perturb(poses, n, seed, deg=2.0, shift=0.04):
    """the first n poses right-multiplied by a rotation of ``deg`` about a random axis and a ``shift`` translation"""
    rng = np.random.RandomState(seed)
    out = poses.double().clone()
    for v in range(n):
        axis = rng.randn(3)
        axis /= np.linalg.norm(axis)
        t = rng.randn(3)
        t *= shift / np.linalg.norm(t)
        xi = torch.from_numpy(np.concatenate([axis * np.deg2rad(deg), t]))[None]
        out[v] = PO.corrected(poses[v:v + 1], xi)[0]
    return out


def _image_error(true_poses, est_poses, focal, H, pts):
    """mean pixel distance between the projections of ``pts`` under the true and the estimated poses"""
    def project(P):
        P = P.double()
        R, t = P[:, :3, :3], P[:, :3, 3]
        xc = torch.einsum("vji,vpj->vpi", R, pts[None] - t[:, None, :])       # R^T (X - t)
        u = focal * xc[..., 0] / -xc[..., 2] + H * 0.5
        v = -focal * xc[..., 1] / -xc[..., 2] + H * 0.5
        return torch.stack([u, v], -1)
    return float((project(true_poses) - project(est_poses)).norm(dim=-1).mean())


def _train(ds, steps, B, refine_mask, pose_lr, warm):
    import b2n
    from b2n import errormap
    from src.core import NeuralField
    from src.renderer import render_rays
    V = len(ds)
    torch.manual_seed(0)
    model = NeuralField(SCENE_CFG).to(DEV).train()
    refine = b2n.PoseRefinement(V, refine=refine_mask) if refine_mask is not None else None
    groups = [{"params": list(model.parameters()), "lr": 1e-2, "weight_decay": 1e-5}]
    if refine is not None:
        groups.append({"params": list(refine.parameters()), "lr": 0.0, "weight_decay": 0.0})
    opt = torch.optim.AdamW(groups)
    gen = torch.Generator(device=DEV).manual_seed(1)
    bg = torch.ones(3, device=DEV)
    for it in range(steps):
        picks = tuple(torch.randint(0, n, (B,), device=DEV, generator=gen) for n in (V, ds.H, ds.W))
        if refine is not None:
            # no pose step while the field is still noise, then a linear decay to 0
            opt.param_groups[1]["lr"] = 0.0 if it < warm else pose_lr * (steps - it) / (steps - warm)
            ro, rd, tgt = refine.rays(ds, picks)
        else:
            ro, rd, tgt = errormap.rays(ds, picks)
        pred = render_rays(model, ro, rd, NEAR, FAR, 64, True, bg_color=bg)[0]
        loss = ((pred - tgt[:, :3]) ** 2).mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    model.eval()
    return model, refine


def _psnr(model, held):
    from src.renderer import render_rays
    ro, rd, tgt = held
    with torch.no_grad():
        pred = torch.cat([render_rays(model, ro[i:i + 2 ** 15], rd[i:i + 2 ** 15], NEAR, FAR, 64, False,
                                      bg_color=torch.ones(3, device=DEV))[0] for i in range(0, ro.shape[0], 2 ** 15)])
    return -10 * math.log10(float(((pred - tgt) ** 2).mean()))


def test_training_recovers_perturbed_poses(tmp_path):
    """100 views of 128^2 of the checker-band sphere; 50 of them stored with a 2 degree rotation about a random axis and
    a 0.04 shift, and only those 50 refined (the 50 exact views fix the gauge).  Joint training at least halves the
    image-plane error of their poses, held-out PSNR is at least that of the same run without refinement, and a control
    run with refinement on exact poses stays under 0.25 px.  The held-out PSNR of the run on exact poses is recorded as
    the reference.  Measured over repeated runs (they differ: the hash-grid scatter uses float atomics): DESIGN.md §5k."""
    import b2n
    from b2n import synthetic
    from src.dataset import BlenderDataset
    V, H, n_bad, steps, B = 100, 128, 50, 3000, 16384
    true = synthetic.hemisphere_poses(V, seed=21)
    stored = _perturb(true, n_bad, seed=5)
    _write_dataset(str(tmp_path / "bad"), true, stored, H)
    _write_dataset(str(tmp_path / "exact"), true, true.double(), H)
    ds_bad = BlenderDataset(str(tmp_path / "bad"), split="train")
    ds_exact = BlenderDataset(str(tmp_path / "exact"), split="train")
    focal = float(ds_bad.focal)
    held_poses = synthetic.hemisphere_poses(8, seed=22)
    ro, rd = zip(*(synthetic.image_rays(p, H=H, W=H) for p in held_poses))
    ro, rd = torch.cat(ro).to(DEV), torch.cat(rd).to(DEV)
    held = (ro, rd, _band_scene(ro, rd))
    g = torch.Generator().manual_seed(7)
    dirs = torch.randn(256, 3, generator=g, dtype=torch.float64)
    pts = RADIUS * dirs / dirs.norm(dim=-1, keepdim=True)
    mask = torch.arange(V) < n_bad
    pose_lr, warm = 2e-3, 300
    prev = b2n.mlp_precision()
    b2n.set_mlp_precision("bf16")
    try:
        m_ref, refine = _train(ds_bad, steps, B, mask, pose_lr, warm)
        m_fix, _ = _train(ds_bad, steps, B, None, pose_lr, warm)
        m_exact, control = _train(ds_exact, steps, B, mask, pose_lr, warm)
        psnr_ref, psnr_fix, psnr_exact = _psnr(m_ref, held), _psnr(m_fix, held), _psnr(m_exact, held)
        with torch.no_grad():
            est = refine.corrected_poses(ds_bad.poses.to(DEV)).cpu()
            est_c = control.corrected_poses(ds_exact.poses.to(DEV)).cpu()
    finally:
        b2n.set_mlp_precision(prev)
    err_before = _image_error(true[:n_bad], ds_bad.poses[:n_bad], focal, H, pts)
    err_after = _image_error(true[:n_bad], est[:n_bad], focal, H, pts)
    err_control = _image_error(true[:n_bad], est_c[:n_bad], focal, H, pts)
    assert torch.equal(est[n_bad:], ds_bad.poses[n_bad:])                 # views outside the mask keep their pose
    record("pose training: image-plane error of the perturbed poses (px)", err_before)
    record("pose training: image-plane error after refinement (px)", err_after)
    record("pose training: image-plane error, control run on exact poses (px)", err_control)
    record("pose training: held-out PSNR with refinement (dB)", psnr_ref)
    record("pose training: held-out PSNR without refinement (dB)", psnr_fix)
    record("pose training: held-out PSNR of the control run on exact poses (dB)", psnr_exact)
    assert err_after <= 0.5 * err_before, (err_before, err_after)
    assert psnr_ref >= psnr_fix, (psnr_ref, psnr_fix)
    assert err_control < 0.25, err_control
    b2n.check_errors()
