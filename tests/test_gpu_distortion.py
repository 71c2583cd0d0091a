"""GPU tests of the distortion loss (b2n.distortion, b2n_distortion_* of include/b2nerf.h): loss and sigma gradient
against the float64 oracle of _distortion_oracle.py within the rounding of an fp32 scan, dense and compact layouts,
static capacity, CUDA-graph capture and determinism, the training render against render_rays, and training."""
import math

import pytest
import torch

import _distortion_oracle as DO
from _util import record, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
NEAR, FAR = 2.0, 6.0
VANILLA = dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)
INSTANT = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
               per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)


def _rays(B, seed=7):
    from b2n import synthetic
    ro, rd, _ = synthetic.random_rays(B, seed=seed)
    return ro.to(DEV), rd.to(DEV)


def _depths(B, N, seed):
    from b2n import march
    ro, rd = _rays(B, seed=seed)
    u = torch.rand(B, N, device=DEV, generator=torch.Generator(DEV).manual_seed(seed))
    return march.march(ro, rd, NEAR, FAR, N, u).z, rd


def _sigma(kind, B, N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    if kind == "random":
        return torch.empty(B, N, device=DEV).exponential_(0.5, generator=g) * (torch.rand(B, N, device=DEV, generator=g) < 0.6)
    if kind == "zero":
        return torch.zeros(B, N, device=DEV)
    if kind == "onehot":
        s = torch.zeros(B, N, device=DEV)
        s[torch.arange(B, device=DEV), torch.randint(0, N, (B,), device=DEV, generator=g)] = 1e4
        return s
    if kind == "huge":                                      # alpha = 1 everywhere: T underflows to 0 in fp32
        return 1e8 * (1.0 + torch.rand(B, N, device=DEV, generator=g))
    raise ValueError(kind)


def _pack(mask):
    """bool [B,N] -> (mask_words int32 [B,W], ray_offset int32 [B+1]) in the layout of b2n_march_mask / _scan"""
    B, N = mask.shape
    W = (N + 31) // 32
    pad = torch.zeros(B, W * 32, dtype=torch.int64, device=mask.device)
    pad[:, :N] = mask.long()
    words = (pad.view(B, W, 32) << torch.arange(32, device=mask.device)).sum(-1)
    words = ((words + 2 ** 31) % 2 ** 32 - 2 ** 31).to(torch.int32)
    off = torch.zeros(B + 1, dtype=torch.int64, device=mask.device)
    off[1:] = torch.cumsum(mask.long().sum(-1), 0)
    return words.contiguous(), off.to(torch.int32)


def _run(sigma_in, z, rd, g_loss, mask_words=None, ray_offset=None):
    import b2n
    s = sigma_in.detach().clone().requires_grad_(True)
    loss = b2n.distortion(s, z, rd, NEAR, FAR, mask_words=mask_words, ray_offset=ray_offset)
    g, = torch.autograd.grad(loss, s, g_loss)
    return loss.detach(), g


def _check(tag, loss, g, sigma_dense, z, rd, g_loss, mask=None):
    """loss [B] and g_sigma (dense [B*N] or the active samples of ``mask``) against the oracle on the dense sigma"""
    B, N = z.shape
    L64, g64 = DO.loss_and_grad(sigma_dense, z, rd, NEAR, FAR, g_loss)
    lb, gb = DO.fp32_bounds(sigma_dense, z, rd, NEAR, FAR, g_loss)
    if mask is not None:
        g64, gb = g64[mask], gb[mask]
    g64, gb = g64.reshape(-1), gb.reshape(-1)
    assert torch.isfinite(loss).all() and torch.isfinite(g).all(), tag
    rl = float(((loss.double() - L64).abs() / lb).max())
    rg = float(((g.double().reshape(-1) - g64).abs() / gb).max()) if g64.numel() else 0.0
    record(f"distortion {tag}: |loss - oracle| / fp32-scan bound", rl)
    record(f"distortion {tag}: |g_sigma - oracle| / fp32-scan bound", rg)
    assert rl <= 1.0 and rg <= 1.0, (tag, rl, rg)


@pytest.mark.parametrize("kind", ["random", "zero", "onehot", "huge"])
@pytest.mark.parametrize("N", [1, 2, 31, 32, 33, 64, 65, 128, 1024])
def test_matches_oracle_dense_and_compact(N, kind):
    """the bound is fp32_bounds of the oracle: 8 * 2^-24 times the sensitivity of each result to one rounding per
    operation of the fp32 scans (the composite's weights, the prefix sums, the reverse scan)"""
    B = 64 if N == 1024 else 512
    z, rd = _depths(B, N, seed=N)
    sigma = _sigma(kind, B, N, seed=N + 1)
    g_loss = torch.randn(B, device=DEV, generator=torch.Generator(DEV).manual_seed(3))
    loss, g = _run(sigma.reshape(-1), z, rd, g_loss)
    _check(f"dense {kind}", loss, g, sigma, z, rd, g_loss)
    if kind == "zero":
        assert torch.equal(loss, torch.zeros_like(loss)) and torch.equal(g, torch.zeros_like(g))
    mask = torch.rand(B, N, device=DEV, generator=torch.Generator(DEV).manual_seed(5)) < 0.5
    mask[: B // 8] = False                                     # rays without an active sample
    words, off = _pack(mask)
    loss_c, g_c = _run(sigma[mask], z, rd, g_loss, words, off)
    _check(f"compact {kind}", loss_c, g_c, sigma * mask, z, rd, g_loss, mask)
    assert torch.equal(loss_c[: B // 8], torch.zeros(B // 8, device=DEV))


@pytest.mark.parametrize("N", [64, 128, 200])
def test_compact_equals_dense_with_the_masked_sigma_set_to_zero(N):
    B = 2048
    z, rd = _depths(B, N, seed=20 + N)
    sigma = _sigma("random", B, N, seed=N)
    g_loss = torch.randn(B, device=DEV)
    mask = torch.rand(B, N, device=DEV) < 0.3
    words, off = _pack(mask)
    loss_d, g_d = _run((sigma * mask).reshape(-1), z, rd, g_loss)
    loss_c, g_c = _run(sigma[mask], z, rd, g_loss, words, off)
    assert torch.equal(loss_c, loss_d)                       # the same arithmetic: an inactive sample reads sigma = 0
    assert torch.equal(g_c, g_d.view(B, N)[mask])


def test_static_capacity_and_device_row_count():
    import b2n
    from b2n import march, synthetic
    from b2n._lib import active_rows
    B, N, R = 4096, 128, 64
    ro, rd = _rays(B, seed=31)
    u = torch.rand(B, N, device=DEV)
    bits = march.pack_occupancy(synthetic.ball_occupancy(R, 1.5, 1.0).to(DEV))
    m0 = march.march(ro, rd, NEAR, FAR, N, u, bits=bits, R=R, bound=1.5)
    n = m0.n_active
    sigma = torch.rand(n, device=DEV) * 3.0
    g_loss = torch.randn(B, device=DEV)
    ref_loss, ref_g = _run(sigma, m0.z, rd, g_loss, m0.mask_words, m0.ray_offset)
    try:
        march.set_static_capacity(True)
        m = march.march(ro, rd, NEAR, FAR, N, u, bits=bits, R=R, bound=1.5)
    finally:
        march.set_static_capacity(False)
    assert m.n_dev is not None and int(m.n_dev.item()) == n and m.n_active == B * N
    cap = torch.full((B * N,), float("nan"), device=DEV)    # rows behind the count hold garbage
    cap[:n] = sigma
    # as in a training step: the forward inside the count's scope, the backward after it (it re-installs the count)
    s = cap.clone().requires_grad_(True)
    with active_rows(m.n_dev):
        loss = b2n.distortion(s, m.z, rd, NEAR, FAR, m.mask_words, m.ray_offset)
    g, = torch.autograd.grad(loss, s, g_loss)
    assert torch.equal(loss.detach(), ref_loss) and torch.equal(g[:n], ref_g)
    assert torch.equal(g[n:], torch.zeros(B * N - n, device=DEV))          # never written, zero-filled by the op
    # a count below the offsets: the rows behind it count as inactive (sigma = 0) and are not written
    k = n // 2
    s = cap.clone().requires_grad_(True)
    with active_rows(torch.tensor([k], device=DEV, dtype=torch.int32)):
        loss_k = b2n.distortion(s, m.z, rd, NEAR, FAR, m.mask_words, m.ray_offset)
    g_k, = torch.autograd.grad(loss_k, s, g_loss)
    cut = sigma.clone()
    cut[k:] = 0.0
    want_loss, want_g = _run(cut, m0.z, rd, g_loss, m0.mask_words, m0.ray_offset)
    assert torch.equal(loss_k.detach(), want_loss) and torch.equal(g_k[:k], want_g[:k])
    assert torch.equal(g_k[k:], torch.zeros(B * N - k, device=DEV))


def test_cuda_graph_replay_and_determinism():
    import b2n
    B, N = 8192, 128
    z, rd = _depths(B, N, seed=41)
    sigma = _sigma("random", B, N, seed=42).reshape(-1)
    g_loss = torch.randn(B, device=DEV)
    l0, g0 = _run(sigma, z, rd, g_loss)
    l1, g1 = _run(sigma, z, rd, g_loss)
    assert torch.equal(l0, l1) and torch.equal(g0, g1)      # two eager runs: the same bits
    s = sigma.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):                                 # warm-up outside the capture
            loss = b2n.distortion(s, z, rd, NEAR, FAR)
            torch.autograd.grad(loss, s, g_loss)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = b2n.distortion(s, z, rd, NEAR, FAR)
        g, = torch.autograd.grad(loss, s, g_loss)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(loss, l0) and torch.equal(g, g0)
    with torch.no_grad():
        s.mul_(0.5)                                        # new inputs in the captured buffer
    graph.replay()
    torch.cuda.synchronize()
    l2, g2 = _run(sigma * 0.5, z, rd, g_loss)
    assert torch.equal(loss, l2) and torch.equal(g, g2) and not torch.equal(l2, l0)


class _Tap(torch.nn.Module):
    """the model with its outputs kept: what it returned for the samples the render handed to it"""

    def __init__(self, model):
        super().__init__()
        self.model = model
        self.mode = getattr(model, "mode", "unknown")
        self.outs = []

    def forward(self, *args, **kw):
        out = self.model(*args, **kw)
        self.outs.append(out)
        return out


@pytest.mark.parametrize("which", ["vanilla", "instant", "part3"])
def test_training_render_equals_render_rays(which):
    import b2n
    from _util import load
    from b2n import march, synthetic
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    torch.manual_seed(0)
    if which == "part3":
        gld = load("field_part3_instant")
        model = NeuralField(gld["cfg"])
        model.load_state_dict(gld["sd"])
    else:
        model = NeuralField(VANILLA if which == "vanilla" else INSTANT)
    model = model.to(DEV).train()
    B, N, R = 1024, 64, 32
    ro, rd = _rays(B, seed=51)
    j = torch.rand(B, N, device=DEV)
    times = torch.rand(B, 1, device=DEV) if which == "part3" else None
    grid = DensityGrid(resolution=R, bound=1.5).to(DEV)
    grid.binary_grid = synthetic.ball_occupancy(R, 1.5, 1.0).to(DEV)
    target = torch.rand(B, 3, device=DEV)
    params = [p for p in model.parameters() if p.requires_grad]

    def mse(color):
        return ((color - target) ** 2).mean()

    tap_ref, tap = _Tap(model), _Tap(model)
    ref = render_rays(tap_ref, ro, rd, NEAR, FAR, N, True, density_grid=grid, times=times, _jitter=j)
    out = b2n.render_rays_distortion(tap, ro, rd, NEAR, FAR, N, True, density_grid=grid, times=times, _jitter=j)
    assert len(out) == len(ref) + 1
    for a, b in zip(out[:3], ref[:3]):
        assert torch.equal(a, b)
    dist = out[3]
    if times is not None:
        assert isinstance(out[4], dict) and out[4].keys() == ref[3].keys()
        for k in ref[3]:
            assert torch.equal(out[4][k], ref[3][k])
    # the distortion is b2n.distortion on the same samples
    m = march.march(ro, rd, NEAR, FAR, N, j, bits=grid.bits(), R=R, bound=1.5, times=times)
    sigma = tap.outs[0][1]
    assert torch.equal(m.z, march.march(ro, rd, NEAR, FAR, N, j, bits=grid.bits(), R=R, bound=1.5).z)
    with torch.no_grad():
        assert torch.equal(dist, b2n.distortion(sigma, m.z, rd, NEAR, FAR, m.mask_words, m.ray_offset))
    if which != "vanilla":                      # softplus densities: every ray with an active sample has weight
        has = (m.ray_offset[1:] > m.ray_offset[:-1])
        assert bool(has.any()) and bool((dist.detach()[has] > 0).all())
        assert bool((dist.detach()[~has] == 0).all())
    # lambda = 0: the same gradients.  At the model's outputs bitwise; the parameter gradients of the hash grids come
    # from float atomics, whose order differs between two backward passes, so they agree to that order only
    outs_ref = [t for t in tap_ref.outs[0] if t.requires_grad]
    outs = [t for t in tap.outs[0] if t.requires_grad]
    assert len(outs) == len(outs_ref) >= 2
    g_ref = torch.autograd.grad(mse(ref[0]), outs_ref + params, allow_unused=True)
    g_out = torch.autograd.grad(mse(out[0]) + 0.0 * dist.mean(), outs + params, allow_unused=True)
    for a, b in zip(g_out[:len(outs)], g_ref[:len(outs)]):
        assert torch.equal(a, b)
    for a, b in zip(g_out[len(outs):], g_ref[len(outs):]):
        assert (a is None) == (b is None)
        if a is not None:
            assert record(f"render_rays_distortion [{which}] lambda = 0: parameter-gradient rel err", rel_err(a, b)) < 2e-5
    b2n.check_errors()


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


def _train(lam, steps=400, B=4096, N=64):
    import b2n
    from b2n import synthetic
    from src.core import NeuralField
    torch.manual_seed(0)
    model = NeuralField(INSTANT).to(DEV).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-5)
    for step in range(1, steps + 1):
        ro, rd, _ = (t.to(DEV) for t in synthetic.random_rays(B, seed=step))
        u = torch.rand(B, N, device=DEV, generator=torch.Generator(DEV).manual_seed(step))
        color, _, _, dist = b2n.render_rays_distortion(model, ro, rd, NEAR, FAR, N, True, _jitter=u)
        loss = torch.nn.functional.mse_loss(color, _sphere_targets(ro, rd)) + lam * dist.mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    model.eval()
    ro, rd, _ = (t.to(DEV) for t in synthetic.random_rays(16384, seed=9999))
    with torch.no_grad():
        color, _, _, dist = b2n.render_rays_distortion(model, ro, rd, NEAR, FAR, N, False)
    psnr = -10 * math.log10(float(((color - _sphere_targets(ro, rd)) ** 2).mean()))
    b2n.check_errors()
    return psnr, float(dist.mean())


def test_training_with_the_distortion_term():
    """the Instant model on the analytic sphere, the same seeds with lambda = 0 and lambda = 0.01 (mip-NeRF 360's)"""
    psnr0, dist0 = _train(0.0)
    psnr1, dist1 = _train(0.01)
    record("distortion training lambda = 0: held-out PSNR (dB)", psnr0)
    record("distortion training lambda = 0.01: held-out PSNR (dB)", psnr1)
    record("distortion training lambda = 0: held-out mean distortion", dist0)
    record("distortion training lambda = 0.01: held-out mean distortion", dist1)
    assert psnr0 > 20.0 and psnr1 > 20.0, (psnr0, psnr1)
    assert dist1 < dist0, (dist0, dist1)
    assert psnr1 >= psnr0 - 1.0, (psnr0, psnr1)
