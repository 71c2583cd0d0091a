"""CPU checks of the error-map contract: the float64 / integer oracle of _errormap_oracle.py against a direct statement
of the update and of the sampling probability p (the oracle's sampler enumerated over a grid of uniforms on tiny maps,
no random draws), and the argument checks of the native and the Python layer, which refuse bad input before any
launch."""
import numpy as np
import pytest
import torch

import _errormap_oracle as EO

# (V, H, W, Hm, Wm): H not divisible by Hm, cells of 2 and 3 pixels; one pixel per cell; one cell per view
MAPS = [(2, 7, 5, 3, 2), (3, 4, 6, 4, 6), (2, 5, 3, 1, 1)]


def _map(kind, V, Hm, Wm, seed=0):
    rng = np.random.RandomState(seed)
    if kind == "unobserved":
        return np.full((V, Hm, Wm), -1.0, np.float32)
    e = rng.rand(V, Hm, Wm).astype(np.float32)
    e[rng.rand(V, Hm, Wm) < 0.3] = 0.0                      # zero-weight cells
    e[rng.rand(V, Hm, Wm) < 0.2] = -1.0                     # never observed
    if e.max() <= 0:
        e.flat[0] = 0.5
    return e


def _enumerate(e, lam, H, W, M0=20000):
    """the oracle sampler's probability of every pixel, from uniforms at the midpoints of a grid: u0 on M0 points,
    (u1, u2) on M1 x M1 points, M1 the least common multiple of every cell's row and column count (exact in a cell)"""
    V, Hm, Wm = e.shape
    sizes = [hi - lo for lo, hi in (EO.cell_bounds(H, Hm), EO.cell_bounds(W, Wm))]
    M1 = int(np.lcm.reduce(np.concatenate(sizes)))
    g0 = (np.arange(M0) + 0.5) / M0
    g1 = (np.arange(M1) + 0.5) / M1
    u = np.stack(np.meshgrid(g0, g1, g1, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)
    v, y, x, r = EO.sample(e, EO.cdf(e), u, lam, H, W)
    hist = np.bincount((v * H + y) * W + x, minlength=V * H * W) / u.shape[0]
    return hist.reshape(V, H, W), (v, y, x, r)


@pytest.mark.parametrize("dims", MAPS, ids=lambda d: "x".join(map(str, d)))
@pytest.mark.parametrize("lam", [0.0, 0.25, 1.0])
@pytest.mark.parametrize("kind", ["observed", "unobserved"])
def test_oracle_sampler_draws_p(dims, lam, kind):
    V, H, W, Hm, Wm = dims
    e = _map(kind, V, Hm, Wm, seed=H * W)
    p = EO.prob(e, lam, H, W)
    assert abs(p.sum() - 1.0) < 1e-12
    hist, (v, y, x, r) = _enumerate(e, lam, H, W)
    # each pixel's u0-interval is off by at most one grid step at each end
    assert np.abs(hist - p).max() <= 2.0 / 20000 + 1e-12, np.abs(hist - p).max()
    assert ((v >= 0) & (v < V) & (y >= 0) & (y < H) & (x >= 0) & (x < W)).all()
    if kind == "unobserved" or lam == 1.0:
        np.testing.assert_allclose(p, 1.0 / (V * H * W), rtol=1e-12)
        assert (r == 1.0).all()
    # the ratio makes a loss unbiased: sum over pixels of p * ratio / N = 1, and ratio = 1 / (N p) pixel by pixel
    np.testing.assert_allclose(r, 1.0 / (V * H * W * p[v, y, x]), rtol=1e-7)
    if lam == 0.0 and kind == "observed":
        w = EO.weights(e)
        cells = EO.cell_of(v, y, x, H, W, Hm, Wm)
        assert (w[cells] > 0).all()                          # the map branch never picks a cell of weight 0


def test_cell_partition():
    for H, Hm in ((7, 3), (800, 128), (5, 5), (5, 1), (129, 128)):
        lo, hi = EO.cell_bounds(H, Hm)
        rows = np.arange(H)
        cell = rows * Hm // H
        for i in range(Hm):
            assert (rows[cell == i] == np.arange(lo[i], hi[i])).all()
        n = hi - lo
        assert n.min() >= 1 and n.max() - n.min() <= 1


def test_oracle_cdf_is_a_monotone_prefix_with_flat_zero_steps():
    rng = np.random.RandomState(1)
    for n in (1, 17, 4096, 4097, 3 * 4096 + 5, 100 * 37 * 41):
        e = rng.rand(n).astype(np.float32) * (rng.rand(n) < 0.5)
        e[rng.rand(n) < 0.1] = np.nan
        c = EO.cdf(e)
        w = EO.weights(e)
        np.testing.assert_allclose(c, np.cumsum(w), rtol=1e-12, atol=0)
        d = np.diff(np.concatenate([[0.0], c]))
        assert (d >= 0).all()
        assert (d[w == 0] == 0).all()                        # exactly flat: weight-0 cells own no part of [0, S)


def test_oracle_update_against_a_direct_statement():
    V, H, W, Hm, Wm = 2, 7, 5, 3, 2
    rng = np.random.RandomState(2)
    e = _map("observed", V, Hm, Wm)
    B = 500
    picks = (rng.randint(0, V, B), rng.randint(0, H, B), rng.randint(0, W, B))
    picks[0][:100], picks[1][:100], picks[2][:100] = 1, 6, 4   # many rays in one cell
    err = rng.rand(B).astype(np.float32) * 1.5 - 0.2
    err[rng.rand(B) < 0.05] = np.nan
    err[rng.rand(B) < 0.05] = np.inf
    err[rng.rand(B) < 0.05] = -np.inf
    got = EO.update(e, picks, err, 0.1, H, W)
    for c in range(V * Hm * Wm):
        sel = [i for i in range(B) if EO.cell_of(picks[0][i], picks[1][i], picks[2][i], H, W, Hm, Wm) == c]
        old = e.ravel()[c]
        if not sel:
            assert got.ravel()[c] == old
            continue
        vals = [min(max(float(err[i]), 0.0), 1.0) if np.isfinite(err[i]) else 0.0 for i in sel]
        m = sum(vals) / len(vals)
        want = m if old < 0 else 0.9 * old + 0.1 * m
        assert abs(got.ravel()[c] - want) <= 2.0 ** -24 + 1e-6 * abs(want), (c, got.ravel()[c], want)
    # order independence: the integer sums make the update a function of the multiset of (pick, err)
    perm = rng.permutation(B)
    again = EO.update(e, tuple(p[perm] for p in picks), err[perm], 0.1, H, W)
    assert np.array_equal(got.view(np.uint32), again.view(np.uint32))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


def test_native_errormap_refuses_bad_arguments(lib):
    fake = 256        # never dereferenced: the arguments are checked before any launch

    def acc(**kw):
        a = dict(img_idx=fake, pix_y=fake, pix_x=fake, err=fake, B=16, V=4, H=8, W=8, Hm=4, Wm=4, acc_sum=fake,
                 acc_cnt=fake)
        a.update(kw)
        return list(a.values()) + [None]

    def smp(**kw):
        a = dict(e=fake, cdf=fake, u=fake, B=16, V=4, H=8, W=8, Hm=4, Wm=4, lam=0.25, img_idx=fake, pix_y=fake,
                 pix_x=fake, ratio=fake)
        a.update(kw)
        return list(a.values()) + [None]

    shape_errors = ((dict(V=0), "V, H, W"), (dict(H=0), "V, H, W"), (dict(Hm=0), "Hm <= H"), (dict(Hm=9), "Hm <= H"),
                    (dict(Wm=9), "Wm <= W"), (dict(V=2 ** 17, Hm=128, Wm=128, H=128, W=128), "2\\^31"))
    for kw, msg in shape_errors + ((dict(B=-1), "B < 2\\^31"), (dict(B=2 ** 31), "B < 2\\^31")):
        with pytest.raises(ValueError, match=msg):
            lib.call("b2n_errormap_accumulate", *acc(**kw))
    for name in ("img_idx", "pix_y", "pix_x", "err", "acc_sum", "acc_cnt"):
        with pytest.raises(ValueError, match="null pointer"):
            lib.call("b2n_errormap_accumulate", *acc(**{name: None}))
    lib.call("b2n_errormap_accumulate", *acc(B=0, err=None))            # empty input: a no-op
    for kw, msg in shape_errors + ((dict(B=-1), "negative B"), (dict(lam=-0.1), "uniform_frac"),
                                   (dict(lam=1.5), "uniform_frac"), (dict(lam=float("nan")), "uniform_frac")):
        with pytest.raises(ValueError, match=msg):
            lib.call("b2n_errormap_sample", *smp(**kw))
    for name in ("e", "cdf", "u", "img_idx", "pix_y", "pix_x", "ratio"):
        with pytest.raises(ValueError, match="null pointer"):
            lib.call("b2n_errormap_sample", *smp(**{name: None}))
    lib.call("b2n_errormap_sample", *smp(B=0, u=None))
    for args, msg in (((fake, fake, fake, 0, 4, 4, 0.1), "V, Hm, Wm"), ((fake, fake, fake, 4, 4, 4, 1.5), "beta"),
                      ((fake, fake, fake, 4, 4, 4, float("nan")), "beta"), ((None, fake, fake, 4, 4, 4, 0.1), "null")):
        with pytest.raises(ValueError, match=msg):
            lib.call("b2n_errormap_apply", *args, None)
    for args, msg in (((fake, 4, 0, 4, fake, fake), "V, Hm, Wm"), ((fake, 2 ** 17, 128, 128, fake, fake), "2\\^31"),
                      ((fake, 4, 4, 4, fake, None), "null")):
        with pytest.raises(ValueError, match=msg):
            lib.call("b2n_errormap_cdf", *args, None)
    assert lib.lib.b2n_errormap_scratch(100, 128, 128) == (400 + 1) * 8
    assert lib.lib.b2n_errormap_scratch(0, 128, 128) == 0 and lib.lib.b2n_errormap_scratch(2 ** 17, 128, 128) == 0


def test_python_layer_refuses_bad_arguments(lib):
    import b2n
    from b2n import errormap
    for kw, msg in ((dict(n_views=0), "n_views"), (dict(H=0), "H"), (dict(W=2.5), "W"), (dict(cells=(0, 4)), "cells"),
                    (dict(cells=4), "cells"), (dict(beta=1.5), "beta"), (dict(beta=True), "beta"),
                    (dict(uniform_frac=-0.1), "uniform_frac"), (dict(n_views=2 ** 17, H=128, W=128), "2\\^31"),
                    (dict(device="cpu"), "no CPU path")):
        args = dict(n_views=4, H=8, W=8)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            b2n.ErrorMap(**args)
    picks = tuple(torch.zeros(4, dtype=torch.int64) for _ in range(3))
    with pytest.raises(ValueError, match="no CPU path"):
        errormap.rays(object(), picks)
    with pytest.raises(ValueError, match="tuple"):
        errormap.rays(object(), picks[:2])
