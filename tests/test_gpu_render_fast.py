"""GPU tests of fast inference rendering (b2n.render, b2n_render_* of include/b2nerf.h): with t_min = 0 it equals the
reference-semantics render_image / render_rays (with and without an occupancy grid, static and dynamic models, both
precision modes); the result does not depend on how samples are grouped into waves; the termination rule matches the
float64 oracle of _render_oracle.py sample for sample; with t_min > 0 it stays within the documented bound while
evaluating fewer samples; and bad input is refused with the model's mode left as it was."""
import contextlib
import math

import numpy as np
import pytest
import torch

import _render_oracle as RO
from _util import record

pytestmark = pytest.mark.gpu
DEV = "cuda"
NEAR, FAR = 2.0, 6.0
SPHERE_CFG = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
                  per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
C2_CFG = dict(mode="part2_instant", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
              per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)       # bench.py's C2 model


def _sphere_targets(ro, rd, radius=0.6):
    """white background, a red-to-blue shaded opaque sphere at the origin (as in test_gpu_training.py)"""
    b = (ro * rd).sum(-1)
    c = (ro * ro).sum(-1) - radius ** 2
    disc = b * b - c
    hit = disc > 0
    t = -b - torch.sqrt(disc.clamp_min(0))
    n = (ro + rd * t[:, None]) / radius
    col = torch.stack([0.5 + 0.5 * n[:, 2], 0.2 + 0.0 * n[:, 0], 0.5 - 0.5 * n[:, 2]], -1)
    return torch.where(hit[:, None], col, torch.ones_like(col))


@contextlib.contextmanager
def _precision(mode):
    import b2n
    prev = b2n.mlp_precision()
    b2n.set_mlp_precision(mode)
    try:
        yield
    finally:
        b2n.set_mlp_precision(prev)


@pytest.fixture(scope="module")
def sphere():
    """an Instant model trained on the analytic sphere for 600 steps of 2^14 rays, long enough for an opaque surface
    (T reaches 1e-4 inside it), and its DensityGrid, updated from it"""
    from b2n import synthetic
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    with _precision("bf16"):
        torch.manual_seed(0)
        model = NeuralField(SPHERE_CFG).to(DEV).train()
        grid = DensityGrid(resolution=64, bound=1.5, threshold=0.05).to(DEV)
        opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-5)
        for step in range(1, 601):
            ro, rd, _ = (t.to(DEV) for t in synthetic.random_rays(2 ** 14, seed=step))
            pred, _, _ = render_rays(model, ro, rd, NEAR, FAR, 64, True, density_grid=grid,
                                     bg_color=torch.ones(3, device=DEV))
            loss = torch.nn.functional.mse_loss(pred, _sphere_targets(ro, rd))
            opt.zero_grad()
            loss.backward()
            opt.step()
            if step >= 100 and step % 50 == 0:
                model.eval()
                grid.update(model, device=DEV)
                model.train()
        model.eval()
        grid.update(model, device=DEV)
    return model, grid


def _view(n, seed=3):
    from b2n import synthetic
    pose = synthetic.hemisphere_poses(1, seed=seed)[0]
    ro, rd = synthetic.image_rays(pose, H=n, W=n)
    return ro.to(DEV), rd.to(DEV)


def _rays(B, seed=7):
    from b2n import synthetic
    ro, rd, _ = synthetic.random_rays(B, seed=seed)
    return ro.to(DEV), rd.to(DEV)


def _masked_count(ro, rd, N, grid):
    import b2n
    return b2n.march.march(ro, rd, NEAR, FAR, N, None, bits=grid.bits(), R=grid.resolution, bound=grid.bound).n_active


def _assert_close(out, color, depth, acc, tag):
    color, depth, acc = color.detach(), depth.detach(), acc.detach()
    ec = record(f"render_fast {tag}: |color - reference|", (out.color - color).abs().max())
    ea = record(f"render_fast {tag}: |acc - reference|", (out.acc - acc).abs().max())
    ed = record(f"render_fast {tag}: |depth - reference| / far", (out.depth - depth).abs().max() / FAR)
    assert ec <= 1e-5 and ea <= 1e-5 and ed <= 1e-5, (ec, ea, ed)


def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("which", ["untrained_c2", "sphere"])
def test_t_min_zero_without_grid_equals_render_image(request, which, precision):
    import b2n
    from src.core import NeuralField
    from src.renderer import render_image, render_rays
    if which == "sphere":
        model = request.getfixturevalue("sphere")[0]
    else:
        torch.manual_seed(0)
        model = NeuralField(C2_CFG).to(DEV).eval()
    H, N = 64, 64
    ro, rd = _view(H)
    with _precision(precision):
        img = render_image(model, ro.view(H, H, 3), rd.view(H, H, 3), NEAR, FAR, N, 1024, True)
        color, depth, acc = render_rays(model, ro, rd, NEAR, FAR, N, False)
        out = b2n.render_image_fast(model, ro.view(H, H, 3), rd.view(H, H, 3), NEAR, FAR, N, t_min=0.0)
    assert out.color.shape == (H, H, 3) and out.depth.shape == (H, H) and out.acc.shape == (H, H)
    assert out.n_evaluated == H * H * N
    assert (out.color - img).abs().max() <= 1e-5
    flat = type(out)(out.color.reshape(-1, 3), out.depth.reshape(-1), out.acc.reshape(-1), 0, 0)
    _assert_close(flat, color, depth, acc, f"no grid {which} {precision}")


@pytest.mark.parametrize("case", ["grid", "grid_bg_per_ray", "empty_grid", "n1"])
def test_t_min_zero_with_grid_equals_masked_render_rays(sphere, case):
    import b2n
    from src.renderer import DensityGrid, render_rays
    model, grid = sphere
    N = 1 if case == "n1" else 96
    if case == "empty_grid":
        grid = DensityGrid(resolution=64, bound=1.5, threshold=0.05).to(DEV)
        grid.binary_grid = torch.zeros(64, 64, 64, dtype=torch.bool, device=DEV)
    ro, rd = _rays(4096)
    bg = torch.rand(ro.shape[0], 3, generator=torch.Generator().manual_seed(1)).to(DEV) \
        if case == "grid_bg_per_ray" else None
    color, depth, acc = render_rays(model, ro, rd, NEAR, FAR, N, False, density_grid=grid, bg_color=bg)
    out = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, bg_color=bg, t_min=0.0)
    _assert_close(out, color, depth, acc, f"grid {case}")
    assert out.n_evaluated == _masked_count(ro, rd, N, grid)
    if case == "empty_grid":
        assert out.n_evaluated == 1                       # sample 0 of ray 0 is evaluated anyway
    if case == "n1":
        bgv = torch.ones(3, device=DEV)
        assert torch.equal(out.color, bgv.expand_as(out.color)) and not out.acc.any()


@pytest.mark.parametrize("t_min", [0.0, 1e-4])
def test_waves_do_not_change_a_bit(sphere, t_min):
    import b2n
    model, grid = sphere
    N = 128
    ro, rd = _rays(8192, seed=11)
    runs = {k: b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, t_min=t_min, _samples_per_wave=k)
            for k in (1, 3, 8, N)}
    runs["policy"] = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, t_min=t_min)
    runs["again"] = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, t_min=t_min)
    ref = runs[1]
    for k, o in runs.items():
        for a, b in ((o.color, ref.color), (o.depth, ref.depth), (o.acc, ref.acc)):
            assert torch.equal(_bits(a), _bits(b)), k
    assert runs[1].n_waves > runs[8].n_waves > runs[N].n_waves >= 1
    if t_min == 0.0:
        assert all(o.n_evaluated == ref.n_evaluated for o in runs.values())


class _Balls(torch.nn.Module):
    """constant sigma inside two balls, 0 outside; colour a smooth function of position in [0, 1].  Evaluated in
    float64 from the fp32 points, so the GPU and the CPU see the same field.  Records the (x, y) of every point."""
    BALLS = ((0.0, 0.0, 0.0, 0.8), (0.5, 0.3, 0.9, 0.4))

    def __init__(self, sigma):
        super().__init__()
        self.sigma = float(sigma)
        self.seen = []

    def forward(self, x, d):
        xd = x.double()
        inside = torch.zeros(x.shape[0], dtype=torch.bool, device=x.device)
        for cx, cy, cz, r in self.BALLS:
            c = torch.tensor([cx, cy, cz], dtype=torch.float64, device=x.device)
            inside |= ((xd - c) ** 2).sum(-1) < r * r
        sigma = torch.where(inside, self.sigma, 0.0).float()[:, None]
        rgb = (0.5 + 0.5 * torch.sin(3.0 * xd + torch.tensor([0.0, 2.0, 4.0], dtype=torch.float64,
                                                               device=x.device))).float()
        self.seen.append(x[:, :2].clone())
        return rgb, sigma


def test_termination_rule_against_oracle():
    """Axis-parallel rays (|d| = 1) through two balls of one constant sigma: every in-ball sample multiplies T by
    q = exp(-sigma*delta), so T takes values near q^k and eps = q^26.5 sits between two of them -- no ray's T comes
    within 1 % of eps, so no tie decides where a ray stops.  With one sample per wave, the samples the model sees per
    ray are exactly the composited ones."""
    import b2n
    N, near, far, n = 128, 1.0, 5.0, 48
    zb = b2n.march.z_tables(near, far, N, DEV)[0]
    delta = (far - near) / (N - 1)
    step = 0.35
    field = _Balls(step / delta)
    eps = math.exp(-step * 26.5)
    ax = torch.linspace(-1.15, 1.15, n)
    gx, gy = torch.meshgrid(ax, ax, indexing="ij")
    ro = torch.stack([gx.reshape(-1), gy.reshape(-1), torch.full((n * n,), -3.0)], -1).contiguous()
    rd = torch.tensor([0.0, 0.0, 1.0]).expand(n * n, 3).contiguous()
    B = ro.shape[0]

    pts = (ro[:, None, :] + rd[:, None, :] * zb.cpu()[None, :, None]).reshape(-1, 3)       # fp32, rounded per op
    with torch.no_grad():
        rgb, sigma = field(pts, None)
    field.seen.clear()
    bg = np.ones(3)
    color, depth, acc, n_comp, gap = RO.render(sigma.view(B, N).numpy(), rgb.view(B, N, 3).numpy(), zb.cpu().numpy(),
                                               np.ones(B), np.ones((B, N), bool), eps, bg)
    assert gap > 0.01, gap
    assert (n_comp < N).sum() > B // 10 and (n_comp == N).sum() > B // 10      # rays that stop, rays that do not

    out = b2n.render_rays_fast(field, ro.to(DEV), rd.to(DEV), near, far, N, t_min=eps, _samples_per_wave=1)
    seen = torch.cat(field.seen).cpu()
    ray = torch.searchsorted(ax, seen[:, 0].contiguous()) * n + torch.searchsorted(ax, seen[:, 1].contiguous())
    assert torch.equal(torch.stack([ro[ray, 0], ro[ray, 1]], -1), seen)
    per_ray = torch.bincount(ray, minlength=B).numpy()
    assert (per_ray == n_comp).all(), np.flatnonzero(per_ray != n_comp)[:10]
    assert out.n_evaluated == int(n_comp.sum())
    for a, b in ((out.color, color), (out.acc, acc), (out.depth / far, depth / far)):
        err = float((a.double().cpu() - torch.from_numpy(b)).abs().max())
        assert err <= 1e-5, err
        record("render_fast oracle: |fast - float64 oracle|", err)
    policy = b2n.render_rays_fast(field, ro.to(DEV), rd.to(DEV), near, far, N, t_min=eps)
    for a, b in ((policy.color, out.color), (policy.depth, out.depth), (policy.acc, out.acc)):
        assert torch.equal(_bits(a), _bits(b))
    assert policy.n_evaluated >= out.n_evaluated          # larger waves evaluate samples behind the stop too


def test_t_min_error_bound_and_savings(sphere):
    """the bound of the contract, and fewer samples than the masked path: with one sample per wave the evaluated samples
    are exactly the composited ones; the default policy evaluates whole waves, so it may evaluate more of them"""
    import b2n
    model, grid = sphere
    N, t_min, H = 128, 1e-4, 256
    ro, rd = _view(H, seed=5)
    full = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, t_min=0.0)
    masked = _masked_count(ro, rd, N, grid)
    assert full.n_evaluated == masked
    bound = t_min + 1e-5
    for k in (None, 1):
        cut = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, N, density_grid=grid, t_min=t_min, _samples_per_wave=k)
        assert (cut.color - full.color).abs().max() <= bound
        assert (cut.acc - full.acc).abs().max() <= bound
        assert (cut.depth - full.depth).abs().max() <= bound * FAR
        assert cut.n_evaluated <= masked
        record(f"render_fast sphere t_min=1e-4 K={k or 'policy'}: evaluated / masked samples", cut.n_evaluated / masked)
    assert cut.n_evaluated < masked


def test_dynamic_model_with_per_ray_times():
    import b2n
    from b2n import synthetic
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    torch.manual_seed(1)
    model = NeuralField(dict(mode="part4", scene_bound=1.5, log2_hashmap_size=16, deform_n_levels=12,
                             deform_log2_hashmap_size=14)).to(DEV).eval()
    grid = DensityGrid(resolution=48, bound=1.5, threshold=0.01).to(DEV)
    grid.update(model, device=DEV)
    ro, rd, _, t = (x.to(DEV) for x in synthetic.random_rays(2048, seed=3, with_time=True))
    color, depth, acc = render_rays(model, ro, rd, NEAR, FAR, 64, False, density_grid=grid, times=t)[:3]
    out = b2n.render_rays_fast(model, ro, rd, NEAR, FAR, 64, density_grid=grid, times=t, t_min=0.0)
    _assert_close(out, color, depth, acc, "part4 per-ray times")
    assert out.n_evaluated == _masked_count(ro, rd, 64, grid)


class _Boom(torch.nn.Module):
    def forward(self, x, d):
        raise RuntimeError("boom")


def test_refusals_and_training_mode():
    import b2n
    from src.core import NeuralField
    torch.manual_seed(0)
    model = NeuralField(SPHERE_CFG).to(DEV).train()
    ro, rd = _rays(64)
    fast = b2n.render_rays_fast
    with pytest.raises(ValueError, match="CUDA"):
        fast(model, ro.cpu(), rd.cpu(), NEAR, FAR, 32)
    with pytest.raises(ValueError, match=r"\[B,3\]"):
        fast(model, ro, rd[:32], NEAR, FAR, 32)
    with pytest.raises(ValueError, match=r"\[B,3\]"):
        fast(model, ro[:, :2], rd[:, :2], NEAR, FAR, 32)
    with pytest.raises(ValueError, match=r"\[H,W,3\]"):
        b2n.render_image_fast(model, ro, rd, NEAR, FAR, 32)
    for n in (0, 1025):
        with pytest.raises(ValueError, match="n_samples"):
            fast(model, ro, rd, NEAR, FAR, n)
    for bad in (-1e-6, 1.0, 1.5, float("nan"), float("inf")):
        with pytest.raises(ValueError, match="t_min"):
            fast(model, ro, rd, NEAR, FAR, 32, t_min=bad)
    with pytest.raises(ValueError, match="bg_color"):
        fast(model, ro, rd, NEAR, FAR, 32, bg_color=torch.ones(5, 3, device=DEV))
    assert model.training
    fast(model, ro, rd, NEAR, FAR, 32)
    assert model.training
    model.eval()
    fast(model, ro, rd, NEAR, FAR, 32)
    assert not model.training
    boom = _Boom().train()
    with pytest.raises(RuntimeError, match="boom"):
        fast(boom, ro, rd, NEAR, FAR, 32)
    assert boom.training
