"""GPU tests of hierarchical importance sampling (b2n.importance, b2n_importance_sample of include/b2nerf.h): the sampler
against the float64 oracle of _importance_oracle.py within the rounding of an fp32 CDF, its exact properties (sorted,
inside the bins, a stable merge, deterministic, capturable in a CUDA graph), the coarse pass against render_rays, the
reuse of the coarse outputs against evaluating the model on every merged sample, training, and the image path."""

import numpy as np
import pytest
import torch

import _importance_oracle as IO
from _util import load, record, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda"
NEAR, FAR = 2.0, 6.0
VANILLA = dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)
INSTANT = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
               per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
TRAIN_STEPS = 400
RADIUS = 1.2


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


class _precision:
    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        import b2n
        self.prev = b2n.mlp_precision()
        b2n.set_mlp_precision(self.mode)

    def __exit__(self, *exc):
        import b2n
        b2n.set_mlp_precision(self.prev)
        return False


def _rays(B, seed=7):
    from b2n import synthetic
    ro, rd, _ = synthetic.random_rays(B, seed=seed)
    return ro.to(DEV), rd.to(DEV)


@pytest.fixture(scope="module")
def trained():
    """the vanilla (C1) model trained on the analytic sphere with hierarchical 64 + 128 sampling, in the pattern of
    test_vanilla_nerf_tcgen05_learns_a_sphere, on the radius-1.2 sphere of test_precision_modes_agree_on_test_view_psnr
    (on the small one the 8x256 net first learns "all white": sigma = relu(.) dies); returns (model, losses)"""
    import b2n
    from b2n import synthetic
    from src.core import NeuralField
    with _precision("bf16"):
        torch.manual_seed(0)
        model = NeuralField(VANILLA).to(DEV).train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        losses = []
        for step in range(1, TRAIN_STEPS + 1):
            ro, rd, _ = (t.to(DEV) for t in synthetic.random_rays(2048, seed=step))
            target = _sphere_targets(ro, rd, RADIUS)
            out = b2n.render_rays_hierarchical(model, ro, rd, NEAR, FAR, 64, 128, True, white_bkgd=True)
            loss = torch.nn.functional.mse_loss(out.color, target)
            coarse = torch.nn.functional.mse_loss(out.coarse_color, target)
            opt.zero_grad()
            (loss + coarse).backward()
            opt.step()
            losses.append(float(loss.detach()))
    model.eval()
    return model, losses


def _sigma(kind, B, Nc, request):
    g = torch.Generator(device=DEV).manual_seed(Nc)
    if kind == "random":
        return torch.empty(B, Nc, device=DEV).exponential_(0.5, generator=g) * (torch.rand(B, Nc, device=DEV, generator=g) < 0.6)
    if kind == "zero":
        return torch.zeros(B, Nc, device=DEV)
    if kind == "onehot":
        s = torch.zeros(B, Nc, device=DEV)
        s[torch.arange(B, device=DEV), torch.randint(0, Nc, (B,), device=DEV, generator=g)] = 1e4
        return s
    raise ValueError(kind)


def _check_sampler(sigma, z, rd, Nf, U, tag):
    """one call of the sampler against the oracle and its exact properties"""
    from b2n.importance import importance_sample
    B, Nc = z.shape
    zf, zm, src = importance_sample(sigma, z, rd, Nf, U)
    zf2, zm2, src2 = importance_sample(sigma, z, rd, Nf, U)
    assert torch.equal(zf, zf2) and torch.equal(zm, zm2) and torch.equal(src, src2)        # deterministic
    # exact properties
    mids32 = 0.5 * (z[:, 1:] + z[:, :-1])
    assert (zf[:, 1:] >= zf[:, :-1]).all()
    assert (zf >= mids32[:, :1]).all() and (zf <= mids32[:, -1:]).all()
    assert (zm[:, 1:] >= zm[:, :-1]).all()
    srcl = src.long()
    assert torch.equal(torch.sort(srcl, -1).values, torch.arange(Nc + Nf, device=DEV).expand(B, -1))   # a permutation
    assert torch.equal(zm, torch.gather(torch.cat([z, zf], -1), 1, srcl))                              # bitwise sources
    tie = zm[:, 1:] == zm[:, :-1]
    assert (srcl[:, 1:] > srcl[:, :-1])[tie].all()          # stable: coarse (s < Nc) before fine, each in its own order
    # the oracle, with the kernel's u (linspace: exactly; stratified: (k + U) / Nf, within 2^-24 of it)
    z64, s64 = z.double().cpu().numpy(), sigma.double().cpu().numpy()
    dn = rd.double().norm(dim=-1).cpu().numpy()
    if U is None:
        u = np.broadcast_to(torch.linspace(0, 1, Nf).double().numpy(), (B, Nf))
    else:
        u = IO.u_stratified(U.double().cpu().numpy())
    mids = 0.5 * (z64[:, 1:] + z64[:, :-1])
    cdf = IO.cdf_of(IO.weights(s64, z64, dn))
    zo, denom, width = IO.invert(cdf, mids, u)
    eps = 8 * Nc * 2.0 ** -24                                 # the rounding of an fp32 CDF
    # the flat-bin rule flips where an fp32 denom (absolute error ~ 16 ulp of 1) crosses 1e-5
    lo, hi = IO.bracket(cdf, mids, u, eps, flat_rel=16 * 2.0 ** -24 / 1e-5)
    ulp = 4 * np.spacing(np.float32(FAR)).astype(np.float64)
    got = zf.double().cpu().numpy()
    assert ((got >= lo - ulp) & (got <= hi + ulp)).all(), tag
    bound = np.abs(width) * eps / np.maximum(denom, 1e-5) + ulp
    smooth = (hi - lo) <= 2 * bound                           # away from a breakpoint of the CDF
    ratio = float((np.abs(got - zo) / bound)[smooth].max())
    record(f"importance sampler {tag}: |z_fine - oracle| / fp32 CDF bound (away from breakpoints)", ratio)
    assert ratio <= 1.0, (tag, ratio)
    zmo, srco = IO.merge(z64, got)
    assert np.array_equal(srco, src.cpu().numpy())
    return zf, zm, src


@pytest.mark.parametrize("det", [True, False], ids=["linspace", "stratified"])
@pytest.mark.parametrize("kind,Nc,Nf", [("random", 64, 128), ("onehot", 64, 128), ("zero", 64, 128),
                                        ("zero", 64, 125), ("random", 3, 1), ("onehot", 3, 5), ("random", 200, 824),
                                        ("random", 33, 96)])
def test_sampler_matches_oracle(kind, Nc, Nf, det, request):
    """zero weights with Nf - 1 a multiple of Nc - 2 (64 + 125) put linspace positions on CDF breakpoints; 200 + 824
    is the compositing limit and needs more than 48 KB of shared memory per block"""
    from b2n import march
    B = 1024
    ro, rd = _rays(B, seed=Nc + Nf)
    U = torch.rand(B, Nc, device=DEV, generator=torch.Generator(device=DEV).manual_seed(1))
    z = march.march(ro, rd, NEAR, FAR, Nc, None if det else U).z
    Uf = None if det else torch.rand(B, Nf, device=DEV, generator=torch.Generator(device=DEV).manual_seed(2))
    _check_sampler(_sigma(kind, B, Nc, request), z, rd, Nf, Uf, f"{kind} {Nc}+{Nf} {'linspace' if det else 'stratified'}")


@pytest.mark.parametrize("det", [True, False], ids=["linspace", "stratified"])
def test_sampler_on_trained_sphere(trained, det):
    import b2n
    from b2n import march
    model = trained[0]
    B, Nc, Nf = 2048, 64, 128
    ro, rd = _rays(B, seed=4242)
    U = None if det else torch.rand(B, Nc, device=DEV)
    m = march.march(ro, rd, NEAR, FAR, Nc, U)
    with torch.no_grad(), _precision("bf16"):
        sigma = model(m.pts, m.dirs)[1].float().reshape(B, Nc)
    assert (sigma > 0).any(-1).float().mean() > 0.05       # the sphere was learnt: the test sees real weight profiles
    _check_sampler(sigma, m.z, rd, Nf, None if det else torch.rand(B, Nf, device=DEV),
                   f"trained sphere {'linspace' if det else 'stratified'}")
    b2n.check_errors()


def test_sampler_captures_into_a_cuda_graph():
    from b2n.importance import importance_sample
    B, Nc, Nf = 4096, 64, 128
    ro, rd = _rays(B)
    from b2n import march
    z = march.march(ro, rd, NEAR, FAR, Nc, torch.rand(B, Nc, device=DEV)).z
    sigma = _sigma("random", B, Nc, None)
    U = torch.rand(B, Nf, device=DEV)
    ref = importance_sample(sigma, z, rd, Nf, U)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        importance_sample(sigma, z, rd, Nf, U)             # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = importance_sample(sigma, z, rd, Nf, U)
    sigma.mul_(0.5)                                        # new inputs in the captured buffers
    U.copy_(torch.rand(B, Nf, device=DEV))
    g.replay()
    torch.cuda.synchronize()
    want = importance_sample(sigma, z, rd, Nf, U)
    for a, b in zip(out, want):
        assert torch.equal(a, b)
    assert not torch.equal(out[0], ref[0])


def _models(request):
    from src.core import NeuralField
    torch.manual_seed(0)
    g = load("field_part3_instant")
    part3 = NeuralField(g["cfg"])
    part3.load_state_dict(g["sd"])
    return {"vanilla": request.getfixturevalue("trained")[0],
            "instant": NeuralField(INSTANT).to(DEV),
            "part3": part3.to(DEV)}


@pytest.mark.parametrize("which", ["vanilla", "instant", "part3"])
def test_coarse_pass_equals_render_rays(which, request):
    import b2n
    from src.renderer import render_rays
    model = _models(request)[which].train()
    B, Nc, Nf = 512, 64, 128
    ro, rd = _rays(B, seed=11)
    j, jf = torch.rand(B, Nc, device=DEV), torch.rand(B, Nf, device=DEV)
    times = torch.rand(B, 1, device=DEV) if which == "part3" else None
    with _precision("bf16"):
        ref = render_rays(model, ro, rd, NEAR, FAR, Nc, True, times=times, _jitter=j)
        out = b2n.render_rays_hierarchical(model, ro, rd, NEAR, FAR, Nc, Nf, True, times=times, _jitter=j,
                                           _jitter_fine=jf)
    for a, b in zip((out.coarse_color, out.coarse_depth, out.coarse_acc), ref[:3]):
        assert torch.equal(a, b)
    model.eval()


@pytest.mark.parametrize("which", ["vanilla", "instant", "part3"])
def test_reuse_equals_evaluating_every_merged_sample(which, request):
    """the fine render reuses the coarse outputs: it must equal the model evaluated on all Nc + Nf merged points and
    composited over the merged depths, forward and in the parameter gradients (fp32 path)"""
    import b2n
    from b2n._lib import call, ptr, stream
    model = _models(request)[which].train()
    B, Nc, Nf = 1024, 64, 128
    ro, rd = _rays(B, seed=12)
    j, jf = torch.rand(B, Nc, device=DEV), torch.rand(B, Nf, device=DEV)
    dyn = which == "part3"
    times = torch.rand(B, 1, device=DEV) if dyn else None
    g_c, g_d, g_a = torch.randn(B, 3, device=DEV), torch.randn(B, device=DEV), torch.randn(B, device=DEV)
    g_x = torch.randn(B, 3, device=DEV)
    params = [p for p in model.parameters() if p.requires_grad]
    with _precision("fp32"):
        out = b2n.render_rays_hierarchical(model, ro, rd, NEAR, FAR, Nc, Nf, True, times=times, _jitter=j,
                                           _jitter_fine=jf)
        loss = (out.color * g_c).sum() + (out.depth * g_d).sum() + (out.acc * g_a).sum()
        if dyn:
            loss = loss + (out.mean_delta_x * g_x).sum()
        grads = torch.autograd.grad(loss, params, allow_unused=True)
        # reference: every merged sample evaluated by the model
        M = Nc + Nf
        z = out.z.detach().contiguous()
        pts, dirs = torch.empty(B * M, 3, device=DEV), torch.empty(B * M, 3, device=DEV)
        tt = torch.empty(B * M, 1, device=DEV) if dyn else None
        call("b2n_march_compact", ptr(ro), ptr(rd), ptr(times), ptr(z), None, None, B, M, None, ptr(pts), ptr(dirs),
             ptr(tt), stream())
        if dyn:
            rgb, sigma, dx = model(pts, dirs, t=tt)
        else:
            (rgb, sigma), dx = model(pts, dirs), None
        color, depth, acc, mdx = b2n.composite(rgb.float(), sigma.float(), z, rd, bg=torch.ones(3, device=DEV),
                                               dx=None if dx is None else dx.float())
        loss_ref = (color * g_c).sum() + (depth * g_d).sum() + (acc * g_a).sum()
        if dyn:
            loss_ref = loss_ref + (mdx * g_x).sum()
        grads_ref = torch.autograd.grad(loss_ref, params, allow_unused=True)
    for name, a, b in (("color", out.color, color), ("depth", out.depth, depth), ("acc", out.acc, acc)) + \
            ((("mean_delta_x", out.mean_delta_x, mdx),) if dyn else ()):
        e = record(f"hierarchical reuse [{which}]: |{name} - all-samples render|", (a.detach() - b.detach()).abs().max())
        assert e <= 1e-5, (name, e)
    worst = 0.0
    for a, b in zip(grads, grads_ref):
        if a is None and b is None:
            continue
        worst = max(worst, rel_err(a, b))
    record(f"hierarchical reuse [{which}]: parameter-gradient rel err", worst)
    assert worst <= 1e-4, worst
    model.eval()


def test_hierarchical_training_learns_the_sphere(trained):
    import b2n
    model, losses = trained
    first, last = sum(losses[:5]) / 5, sum(losses[-20:]) / 20
    record("hierarchical training: last/first loss ratio", last / first)
    ro, rd = _rays(8192, seed=9999)
    target = _sphere_targets(ro, rd, RADIUS)
    hit = (target != 1).any(-1)
    with torch.no_grad(), _precision("bf16"):
        out = b2n.render_rays_hierarchical(model, ro, rd, NEAR, FAR, 64, 128, False)
    psnr = -10 * torch.log10(((out.color - target) ** 2).mean()).item()
    acc_hit = float(out.acc[hit].mean())
    record("hierarchical training: held-out PSNR (dB)", psnr)
    record("hierarchical training: mean acc of the rays that hit the sphere", acc_hit)
    # measured on a B200: loss ratio 0.0175, held-out PSNR 25.3 dB, acc 0.98 on the rays that hit the sphere
    assert last < 0.1 * first, (first, last)
    assert psnr > 20.0, psnr
    assert acc_hit > 0.5, acc_hit                            # geometry was learnt, not an all-white field


def test_render_image_hierarchical_equals_unchunked_and_restores_mode(trained):
    import b2n
    from b2n import synthetic
    model = trained[0]
    H = 24
    pose = synthetic.hemisphere_poses(1, seed=3)[0]
    ro, rd = (t.to(DEV) for t in synthetic.image_rays(pose, H=H, W=H))
    ro, rd = ro.reshape(H, H, 3), rd.reshape(H, H, 3)
    with _precision("bf16"):
        model.train()
        img = b2n.render_image_hierarchical(model, ro, rd, NEAR, FAR, 64, 128, 100, True)      # 576 rays: ragged chunk
        assert model.training
        model.eval()
        with torch.no_grad():
            ref = b2n.render_rays_hierarchical(model, ro.reshape(-1, 3), rd.reshape(-1, 3), NEAR, FAR, 64, 128, False)
    for a, b in zip(img[:7], ref[:7]):
        assert torch.equal(a.reshape(b.shape), b)
    assert img.color.shape == (H, H, 3) and img.z.shape == (H, H, 192) and img.mean_delta_x is None

    class Broken(torch.nn.Module):
        def forward(self, *a, **k):
            raise RuntimeError("broken model")
    bad = Broken().train()
    with pytest.raises(RuntimeError, match="broken model"):
        b2n.render_image_hierarchical(bad, ro, rd, NEAR, FAR, 64, 128, 100, True)
    assert bad.training
    bad.eval()
    with pytest.raises(RuntimeError, match="broken model"):
        b2n.render_image_hierarchical(bad, ro, rd, NEAR, FAR, 64, 128, 100, True)
    assert not bad.training

