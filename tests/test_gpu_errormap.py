"""GPU tests of error-map ray sampling (b2n.errormap, b2n_errormap_* of include/b2nerf.h): the update and the CDF
against the oracle of _errormap_oracle.py bit for bit, the picks and ratios for pinned uniforms, the statistics of
2^22 draws, in-range picks for degenerate uniforms and maps, determinism and CUDA-graph capture, the rays of the picks
against sample_random_rays, training on a scene whose detail is concentrated, and the multi-rank update."""
import os

import numpy as np
import pytest
import torch

import _errormap_oracle as EO
from _util import GOLDEN, record

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _state(emap):
    return emap.e.cpu().numpy().copy(), emap.cdf.cpu().numpy().copy()


def _errors(B, gen):
    err = torch.rand(B, generator=gen) * 1.6 - 0.3                          # negative and > 1 included
    k = torch.randint(0, 12, (B,), generator=gen)
    err[k == 0], err[k == 1], err[k == 2] = float("nan"), float("inf"), -float("inf")
    return err


def _picks(B, V, H, W, gen, hot=0):
    p = [torch.randint(0, n, (B,), generator=gen) for n in (V, H, W)]
    for t, val in zip(p, (V - 1, H - 1, W - 1)):
        t[:hot] = val                                                      # many rays in one cell
    return p


@pytest.mark.parametrize("dims", [(3, 37, 29, 8, 5), (100, 800, 800, 128, 128)], ids=["small", "c2"])
def test_update_and_cdf_match_oracle_bitwise(dims):
    import b2n
    V, H, W, Hm, Wm = dims
    emap = b2n.ErrorMap(V, H, W, cells=(Hm, Wm))
    gen = torch.Generator().manual_seed(V + H)
    e_ref = np.full((V, Hm, Wm), -1.0, np.float32)
    B = 2 ** 18 if V == 100 else 20000
    for step in range(3):
        picks = _picks(B, V, H, W, gen, hot=B // 4)
        err = _errors(B, gen)
        emap.update(tuple(t.to(DEV) for t in picks), err.to(DEV))
        e_ref = EO.update(e_ref, [t.numpy() for t in picks], err.numpy(), 0.1, H, W)
        e, c = _state(emap)
        assert np.array_equal(e.view(np.uint32), e_ref.view(np.uint32)), step
        assert np.array_equal(c.view(np.uint64), EO.cdf(e_ref).view(np.uint64)), step
        assert int(emap.acc_sum.abs().sum()) == 0 and int(emap.acc_cnt.abs().sum()) == 0
    assert (e >= 0).sum() > 0 and (e < 0).sum() > 0 if V == 100 else (e >= 0).all()


def _structured(V, Hm, Wm, seed=0):
    rng = np.random.RandomState(seed)
    e = (rng.rand(V, Hm, Wm) ** 4).astype(np.float32)
    e[:, : Hm // 3] = 0.0                                                  # zero-weight rows
    e[0] = -1.0                                                            # an unobserved view
    e[1, 2, 3] = 1.0                                                       # one hot cell
    return e


def _with_map(e, H, W, lam):
    import b2n
    V, Hm, Wm = e.shape
    emap = b2n.ErrorMap(V, H, W, cells=(Hm, Wm), uniform_frac=lam)
    emap.e.copy_(torch.from_numpy(e))
    emap.rebuild_cdf()
    return emap


def _check_picks_against_oracle(emap, e, u, lam, H, W, tag):
    (v, y, x), r = emap.sample(u.shape[0], u=u)
    c = emap.cdf.cpu().numpy()
    assert np.array_equal(c.view(np.uint64), EO.cdf(e).view(np.uint64))
    vo, yo, xo, ro = EO.sample(e, c, u.cpu().numpy(), lam, H, W)
    v, y, x, r = (t.cpu().numpy() for t in (v, y, x, r))
    V, Hm, Wm = e.shape
    assert ((v >= 0) & (v < V) & (y >= 0) & (y < H) & (x >= 0) & (x < W)).all(), tag
    same = (v == vo) & (y == yo) & (x == xo)
    if not same.all():
        # only where t lies within fp64 rounding of a CDF breakpoint may the neighbouring cell be drawn
        u0 = u[:, 0].double().cpu().numpy()[~same]
        L = float(np.float32(lam))
        t = (u0 - L) / (1 - L) * c[-1]
        cg = EO.cell_of(v[~same], y[~same], x[~same], H, W, Hm, Wm)
        co = EO.cell_of(vo[~same], yo[~same], xo[~same], H, W, Hm, Wm)
        edge = c[np.minimum(cg, co)]
        assert (np.abs(edge - t) <= 1e-12 * c[-1]).all(), tag
    record(f"errormap sample [{tag}]: share of picks off the oracle (breakpoints)", 1.0 - same.mean())
    ok = same & np.isfinite(ro)
    rel = np.abs(r[ok].astype(np.float64) - ro[ok]) / ro[ok]
    record(f"errormap sample [{tag}]: ratio rel err", rel.max())
    assert rel.max() <= 1e-6, tag
    return v, y, x, r


@pytest.mark.parametrize("lam", [0.0, 0.25, 1.0])
@pytest.mark.parametrize("kind", ["structured", "unobserved"])
def test_sample_matches_oracle_for_pinned_u(lam, kind):
    V, H, W, Hm, Wm = 5, 53, 47, 12, 9
    e = _structured(V, Hm, Wm) if kind == "structured" else np.full((V, Hm, Wm), -1.0, np.float32)
    emap = _with_map(e, H, W, lam)
    u = torch.rand(200_000, 3, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3))
    v, y, x, r = _check_picks_against_oracle(emap, e, u, lam, H, W, f"{kind} lam={lam}")
    if kind == "unobserved" or lam == 1.0:
        assert (r == 1.0).all()
    if lam == 0.0 and kind == "structured":
        assert (EO.weights(e)[EO.cell_of(v, y, x, H, W, Hm, Wm)] > 0).all()


def test_statistics_of_many_draws():
    """2^22 draws against p: a chi-square over the pixels (threshold dof + 8 sqrt(2 dof), about 8 sigma, which the
    fixed seed passes with margin), zero draws where p = 0, mean ratio within 5 standard errors of the share of pixels
    with p > 0 (1 for lam > 0); lam = 1 is uniform"""
    V, H, W, Hm, Wm = 4, 48, 40, 12, 10
    e = _structured(V, Hm, Wm, seed=5)
    B = 2 ** 22
    for lam in (0.0, 0.25, 1.0):
        emap = _with_map(e, H, W, lam)
        (v, y, x), r = emap.sample(B, generator=torch.Generator(device=DEV).manual_seed(11))
        obs = torch.bincount((v * H + y) * W + x, minlength=V * H * W).double().cpu().numpy()
        p = EO.prob(e, lam, H, W).ravel()
        exp = p * B
        pos = exp > 0
        assert obs[~pos].sum() == 0, lam
        chi2 = float((((obs - exp) ** 2)[pos] / exp[pos]).sum())
        dof = int(pos.sum()) - 1
        z = (chi2 - dof) / np.sqrt(2 * dof)
        record(f"errormap statistics lam={lam}: chi-square z-score over {dof} dof", abs(z))
        assert chi2 < dof + 8 * np.sqrt(2 * dof), (lam, chi2, dof)
        # E[ratio] = sum over the pixels with p > 0 of p / (N p) = their share of the N pixels: 1 whenever lam > 0;
        # with lam = 0 the pixels of weight-0 cells are never drawn and no weight can stand in for them
        cover = float(pos.mean())
        assert lam == 0.0 or cover == 1.0
        rd = r.double()
        mean, se = float(rd.mean()), float(rd.std() / np.sqrt(B))
        record(f"errormap statistics lam={lam}: |mean ratio - share of p > 0| / standard error",
               abs(mean - cover) / max(se, 1e-30))
        assert abs(mean - cover) <= 5 * se + 1e-6, (lam, mean, cover, se)
        if lam == 1.0:
            assert (r == 1).all()
            np.testing.assert_allclose(p, 1.0 / (V * H * W))


def test_degenerate_uniforms_and_maps_give_in_range_picks():
    V, H, W, Hm, Wm = 3, 11, 13, 4, 5
    vals = torch.tensor([0.0, 1.0, float("nan")])
    u = torch.cartesian_prod(vals, vals, vals).float().to(DEV)              # every combination of 0, 1, NaN
    good = _structured(V, Hm, Wm)
    maps = {"structured": good, "inf": np.full((V, Hm, Wm), np.inf, np.float32),
            "nan": np.full((V, Hm, Wm), np.nan, np.float32), "zero": np.zeros((V, Hm, Wm), np.float32)}
    mixed = good.copy()
    mixed[1, 0, 0], mixed[2, 1, 1] = np.inf, np.nan
    maps["mixed"] = mixed
    for name, e in maps.items():
        for lam in (0.0, 0.25, 1.0):
            emap = _with_map(e, H, W, lam)
            (v, y, x), r = emap.sample(u.shape[0], u=u)
            v, y, x = (t.cpu().numpy() for t in (v, y, x))
            assert ((v >= 0) & (v < V) & (y >= 0) & (y < H) & (x >= 0) & (x < W)).all(), (name, lam)
            vo, yo, xo, _ = EO.sample(e, emap.cdf.cpu().numpy(), u.cpu().numpy(), lam, H, W)
            assert np.array_equal(v, vo) and np.array_equal(y, yo) and np.array_equal(x, xo), (name, lam)


def _loop(emap, us, errs_of):
    out = []
    for u in us:
        picks, r = emap.sample(u.shape[0], u=u)
        emap.update(picks, errs_of(picks))
        out.append((picks, r))
    return out


def _errs_of(picks):
    v, y, x = picks
    return ((v * 131 + y * 7 + x * 3) % 17).float() / 16.0 * 1.1


def test_deterministic_and_graph_capture_equals_eager():
    import b2n
    V, H, W = 6, 64, 48
    B = 2 ** 16
    us = [torch.rand(B, 3, device=DEV, generator=torch.Generator(device=DEV).manual_seed(s)) for s in range(6)]
    runs = []
    for _ in range(2):
        emap = b2n.ErrorMap(V, H, W, cells=(16, 12))
        out = _loop(emap, us, _errs_of)
        runs.append((out, _state(emap)))
    for (a, sa), (b, sb) in zip(runs[0][0], runs[1][0]):
        assert all(torch.equal(p, q) for p, q in zip(a, b)) and torch.equal(sa, sb)
    assert all(np.array_equal(p.view(np.uint8), q.view(np.uint8)) for p, q in zip(runs[0][1], runs[1][1]))
    # capture: one step of sample + update on a static uniform buffer, replayed with new uniforms
    emap = b2n.ErrorMap(V, H, W, cells=(16, 12))
    u_static = us[0].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    warm = b2n.ErrorMap(V, H, W, cells=(16, 12))
    with torch.cuda.stream(s):
        _loop(warm, [u_static], _errs_of)                                  # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        (picks, ratio), = _loop(emap, [u_static], _errs_of)
    for i, u in enumerate(us):
        u_static.copy_(u)
        g.replay()
        ref_picks, ref_ratio = runs[0][0][i]
        assert all(torch.equal(p, q) for p, q in zip(picks, ref_picks)) and torch.equal(ratio, ref_ratio), i
    torch.cuda.synchronize()
    e, c = _state(emap)
    assert np.array_equal(e.view(np.uint32), runs[0][1][0].view(np.uint32))
    assert np.array_equal(c.view(np.uint64), runs[0][1][1].view(np.uint64))


@pytest.mark.parametrize("tag", ["blender", "dynamic"])
def test_rays_of_picks_equal_sample_random_rays(tag):
    import b2n
    from b2n import errormap
    from src.dataset import BlenderDataset, DynamicDataset
    cls = BlenderDataset if tag == "blender" else DynamicDataset
    ds = cls(os.path.join(GOLDEN, "dataset_tiny"), split="train", white_bkgd=True, scene_scale=0.5)
    torch.manual_seed(77)
    ref = ds.sample_random_rays(257, DEV)
    torch.manual_seed(77)
    picks = tuple(t.to(DEV) for t in ds._draw(257, "cpu"))
    out = errormap.rays(ds, picks)
    assert len(out) == len(ref) == (4 if tag == "dynamic" else 3)
    for a, b in zip(out, ref):
        assert torch.equal(a, b)
    # picks of an error map over the dataset: the same kernel on the same resident copies
    emap = b2n.ErrorMap(len(ds), ds.H, ds.W, cells=(6, 5))
    picks, _ = emap.sample(1000, generator=torch.Generator(device=DEV).manual_seed(1))
    out = emap.rays(ds, picks)
    from oracle import nerf_oracle as O
    host = O.sample_rays_host(ds.poses, ds._rgba8, ds._times_tensor(), *(t.cpu() for t in picks), ds.H, ds.W,
                              ds.focal, 0.5)
    assert torch.equal(out[2].cpu(), host[2]) and torch.equal(out[0].cpu(), host[0])
    with pytest.raises(ValueError, match="views"):
        b2n.ErrorMap(len(ds) + 1, ds.H, ds.W).rays(ds, picks)


def test_python_layer_refuses_bad_arguments():
    import b2n
    emap = b2n.ErrorMap(2, 8, 8, cells=(4, 4))
    assert emap.e.shape == (2, 4, 4)
    assert b2n.ErrorMap(2, 8, 6).e.shape == (2, 8, 6)                      # the default 128 x 128, clipped to H x W
    picks, _ = emap.sample(16)
    for bad, msg in ((dict(batch_size=-1), "batch_size"), (dict(batch_size=4, u=torch.rand(4, 2, device=DEV)), "u"),
                     (dict(batch_size=4, u=torch.rand(4, 3)), "no CPU path")):
        with pytest.raises(ValueError, match=msg):
            emap.sample(**bad)
    with pytest.raises(ValueError, match="err"):
        emap.update(picks, torch.rand(16, 1, device=DEV))
    with pytest.raises(ValueError, match="16 rays, expected 8"):
        emap.update(picks, torch.rand(8, device=DEV))
    with pytest.raises(ValueError, match="int64"):
        emap.update(tuple(t.int() for t in picks), torch.rand(16, device=DEV))
    with pytest.raises(ValueError, match="no CPU path"):
        emap.update(picks, torch.rand(16))
    (v, y, x), r = emap.sample(0)
    assert v.shape == (0,) and r.shape == (0,)


# ---- training on a scene whose detail is concentrated
SCENE_CFG = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
                 per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
RADIUS, BAND = 0.6, 0.25


def _band_scene(ro, rd):
    """white background and a red-to-blue shaded sphere (as in test_gpu_render_fast.py), with a black-and-white
    checker of 24 x 6 squares on the latitude band |n_z| < BAND; returns (colour [B,3], on-band mask [B])"""
    b = (ro * rd).sum(-1)
    disc = b * b - ((ro * ro).sum(-1) - RADIUS ** 2)
    hit = disc > 0
    n = (ro + rd * (-b - torch.sqrt(disc.clamp_min(0)))[:, None]) / RADIUS
    col = torch.stack([0.5 + 0.5 * n[:, 2], 0.2 + 0.0 * n[:, 0], 0.5 - 0.5 * n[:, 2]], -1)
    band = hit & (n[:, 2].abs() < BAND)
    az = torch.atan2(n[:, 1], n[:, 0])
    check = ((torch.floor(az * 24 / (2 * np.pi)) + torch.floor(n[:, 2] * 6 / (2 * BAND))) % 2)[:, None].expand(-1, 3)
    col = torch.where(band[:, None], check, col)
    return torch.where(hit[:, None], col, torch.ones_like(col)), band


def _views(V, H, seed):
    from b2n import synthetic
    poses = synthetic.hemisphere_poses(V, seed=seed)
    ro, rd = zip(*(synthetic.image_rays(p, H=H, W=H) for p in poses))
    ro, rd = torch.stack(ro).to(DEV), torch.stack(rd).to(DEV)                # [V, H*H, 3]
    tgt, band = _band_scene(ro.reshape(-1, 3), rd.reshape(-1, 3))
    return ro, rd, tgt.reshape(V, H * H, 3), band.reshape(V, H, H)


def _train(views, H, steps, B, use_map):
    import b2n
    from src.core import NeuralField
    from src.renderer import render_rays
    ro_all, rd_all, tgt_all, _ = views
    V = ro_all.shape[0]
    torch.manual_seed(0)
    model = NeuralField(SCENE_CFG).to(DEV).train()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-5)
    emap = b2n.ErrorMap(V, H, H, cells=(16, 16))
    gen = torch.Generator(device=DEV).manual_seed(1)
    losses = []
    for _ in range(steps):
        if use_map:
            (v, y, x), _ = emap.sample(B, generator=gen)
        else:
            v, y, x = (torch.randint(0, n, (B,), device=DEV, generator=gen) for n in (V, H, H))
        k = y * H + x
        ro, rd, tgt = ro_all[v, k], rd_all[v, k], tgt_all[v, k]
        pred = render_rays(model, ro, rd, 2.0, 6.0, 64, True, bg_color=torch.ones(3, device=DEV))[0]
        per_ray = ((pred - tgt) ** 2).mean(-1)
        loss = per_ray.mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        if use_map:
            emap.update((v, y, x), per_ray.detach())
        losses.append(float(loss.detach()))
    model.eval()
    return model, emap, losses


def _psnr(model, views, mask=None):
    from src.renderer import render_rays
    ro, rd, tgt, band = views
    ro, rd, tgt = ro.reshape(-1, 3), rd.reshape(-1, 3), tgt.reshape(-1, 3)
    with torch.no_grad():
        pred = torch.cat([render_rays(model, ro[i:i + 2 ** 15], rd[i:i + 2 ** 15], 2.0, 6.0, 64, False,
                                      bg_color=torch.ones(3, device=DEV))[0] for i in range(0, ro.shape[0], 2 ** 15)])
    err = ((pred - tgt) ** 2).mean(-1)
    if mask is not None:
        err = err[mask.reshape(-1)]
    return -10 * float(torch.log10(err.mean()))


def test_training_concentrates_the_map_on_the_detail():
    """an Instant model trained on the checker-band sphere with error-map picks (lam = 0.25, unweighted loss, as
    Instant-NGP): the map's mass per pixel is at least 3x higher on the band than on cells without band pixels, the
    training loss falls as with uniform picks, and the PSNR over every training pixel stays within 3 dB of uniform
    sampling's (a quality comparison at a fixed budget is tools/kbench.py errormap)"""
    import b2n
    V, H, steps, B = 48, 64, 300, 4096
    train, held = _views(V, H, seed=21), _views(8, H, seed=22)
    prev = b2n.mlp_precision()
    b2n.set_mlp_precision("bf16")
    try:
        m_map, emap, l_map = _train(train, H, steps, B, True)
        m_uni, _, l_uni = _train(train, H, steps, B, False)
        fit_map, fit_uni = _psnr(m_map, train), _psnr(m_uni, train)
        psnr_map, psnr_uni = _psnr(m_map, held), _psnr(m_uni, held)
        band_map, band_uni = _psnr(m_map, held, held[3]), _psnr(m_uni, held, held[3])
    finally:
        b2n.set_mlp_precision(prev)
    # the map's mass per pixel: cells mostly on the band against cells with no band pixel
    band = train[3].float().reshape(V, 16, H // 16, 16, H // 16).mean((2, 4))
    e = emap.e.clamp_min(0)
    on, off = float(e[band > 0.5].mean()), float(e[band == 0].mean())
    record("errormap training: map mass per pixel, band cells / cells without band", on / max(off, 1e-30))
    record("errormap training: PSNR over all training pixels, error map (dB)", fit_map)
    record("errormap training: PSNR over all training pixels, uniform (dB)", fit_uni)
    record("errormap training: held-out PSNR error map (dB)", psnr_map)
    record("errormap training: held-out PSNR uniform (dB)", psnr_uni)
    record("errormap training: held-out band PSNR error map (dB)", band_map)
    record("errormap training: held-out band PSNR uniform (dB)", band_uni)
    first_m, last_m = np.mean(l_map[:5]), np.mean(l_map[-20:])
    first_u, last_u = np.mean(l_uni[:5]), np.mean(l_uni[-20:])
    record("errormap training: last/first training loss, error map", last_m / first_m)
    record("errormap training: last/first training loss, uniform", last_u / first_u)
    assert on > 3 * off, (on, off)
    assert last_m < 0.3 * first_m and last_u < 0.3 * first_u, (first_m, last_m, first_u, last_u)
    assert fit_map > fit_uni - 3.0, (fit_map, fit_uni)
    b2n.check_errors()


# ---- multi-rank update
def _dp_worker(rank, world, port, out):
    import torch.distributed as dist
    import b2n
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    V, H, W, B = 5, 40, 36, 30000
    gen = torch.Generator().manual_seed(3)
    steps = [(_picks(B * world, V, H, W, gen, hot=B // 2), _errors(B * world, gen)) for _ in range(3)]
    split, whole = b2n.ErrorMap(V, H, W, cells=(9, 7), device=dev), b2n.ErrorMap(V, H, W, cells=(9, 7), device=dev)
    for picks, err in steps:
        sl = slice(rank * B, (rank + 1) * B)
        split.update(tuple(t[sl].to(dev) for t in picks), err[sl].to(dev), group=dist.group.WORLD)
        whole.update(tuple(t.to(dev) for t in picks), err.to(dev))
    same = torch.equal(split.e.view(torch.int32), whole.e.view(torch.int32)) and \
        torch.equal(split.cdf.view(torch.int64), whole.cdf.view(torch.int64))
    flags = torch.tensor([int(same)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if rank == 0:
        torch.save(bool(flags.item()), out)
    dist.barrier(device_ids=[rank])
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_multi_rank_update_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    out = str(tmp_path / "em.pt")
    mp.spawn(_dp_worker, args=(2, 29547, out), nprocs=2, join=True)
    assert torch.load(out)
