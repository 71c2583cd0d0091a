"""CPU checks of the hierarchical-sampling contract: the float64 oracle of _importance_oracle.py against an independent
torch transcription of the original NeRF's raw2outputs weights and sample_pdf (nerf-pytorch, det=True and with sorted
stratified u), and the argument checks of b2n_importance_sample, which refuse bad input before any launch."""
import numpy as np
import pytest
import torch

import _importance_oracle as IO


def _nerf_weights(sigma, z, rays_d):
    """nerf-pytorch raw2outputs: the weights from (relu'd) densities"""
    dists = z[..., 1:] - z[..., :-1]
    dists = torch.cat([dists, torch.tensor([1e10], dtype=z.dtype).expand(dists[..., :1].shape)], -1)
    dists = dists * torch.norm(rays_d[..., None, :], dim=-1)
    alpha = 1.0 - torch.exp(-sigma * dists)
    return alpha * torch.cumprod(torch.cat([torch.ones((alpha.shape[0], 1), dtype=z.dtype), 1.0 - alpha + 1e-10],
                                           -1), -1)[:, :-1]


def _sample_pdf(bins, weights, n_samples, det, u=None):
    """nerf-pytorch sample_pdf; ``u`` replaces the torch.rand draw of det=False"""
    weights = weights + 1e-5
    pdf = weights / torch.sum(weights, -1, keepdim=True)
    cdf = torch.cumsum(pdf, -1)
    cdf = torch.cat([torch.zeros_like(cdf[..., :1]), cdf], -1)
    if det:
        u = torch.linspace(0.0, 1.0, steps=n_samples, dtype=cdf.dtype)
        u = u.expand(list(cdf.shape[:-1]) + [n_samples])
    u = u.contiguous()
    inds = torch.searchsorted(cdf, u, right=True)
    below = torch.max(torch.zeros_like(inds - 1), inds - 1)
    above = torch.min((cdf.shape[-1] - 1) * torch.ones_like(inds), inds)
    inds_g = torch.stack([below, above], -1)
    matched_shape = [inds_g.shape[0], inds_g.shape[1], cdf.shape[-1]]
    cdf_g = torch.gather(cdf.unsqueeze(1).expand(matched_shape), 2, inds_g)
    bins_g = torch.gather(bins.unsqueeze(1).expand(matched_shape), 2, inds_g)
    denom = cdf_g[..., 1] - cdf_g[..., 0]
    denom = torch.where(denom < 1e-5, torch.ones_like(denom), denom)
    t = (u - cdf_g[..., 0]) / denom
    return bins_g[..., 0] + t * (bins_g[..., 1] - bins_g[..., 0])


def _rays(B, Nc, seed, near=2.0, far=6.0):
    rng = np.random.RandomState(seed)
    t = np.linspace(0.0, 1.0, Nc)
    z = near * (1 - t) + far * t
    mids = 0.5 * (z[1:] + z[:-1])
    lo, hi = np.concatenate([z[:1], mids]), np.concatenate([mids, z[-1:]])
    z = lo + (hi - lo) * rng.rand(B, Nc)                                     # jittered strata: sorted per ray
    d = rng.randn(B, 3)
    return z, d


def _sigma(kind, B, Nc, seed):
    rng = np.random.RandomState(seed + 1)
    if kind == "random":
        return rng.exponential(2.0, (B, Nc)) * (rng.rand(B, Nc) < 0.6)
    if kind == "zero":
        return np.zeros((B, Nc))
    s = np.zeros((B, Nc))                                                    # one opaque sample: one-hot weights
    s[np.arange(B), rng.randint(0, Nc, B)] = 1e4
    return s


@pytest.mark.parametrize("Nc,Nf", [(64, 128), (3, 5), (17, 1), (3, 1), (33, 96)])
@pytest.mark.parametrize("kind", ["random", "zero", "onehot"])
@pytest.mark.parametrize("det", [True, False])
def test_oracle_equals_nerf_sample_pdf(Nc, Nf, kind, det):
    B = 48
    z, d = _rays(B, Nc, seed=Nc * 7 + Nf)
    sigma = _sigma(kind, B, Nc, seed=Nc + Nf)
    t = torch.from_numpy
    w_ref = _nerf_weights(t(sigma), t(z), t(d))
    w = IO.weights(sigma, z, np.linalg.norm(d, axis=-1))
    np.testing.assert_allclose(w, w_ref.numpy(), rtol=1e-12, atol=1e-15)
    if kind == "onehot":
        assert (np.abs(w.max(-1) - 1.0) < 1e-7).all() and (np.sort(w, -1)[:, -2] < 1e-7).all()
    if det:
        u = np.broadcast_to(np.linspace(0.0, 1.0, Nf), (B, Nf))
    else:
        u = IO.u_stratified(np.random.RandomState(3).rand(B, Nf))
    zf, cdf, mids = IO.sample(sigma, z, np.linalg.norm(d, axis=-1), u)
    zf_ref = _sample_pdf(t(mids), w_ref[:, 1:-1], Nf, det, u=None if det else t(u))
    # expm1 against 1 - exp and the order of the sums differ in the last bits; where u sits on a breakpoint of the CDF
    # (u = 1 against a last entry rounded below 1, say) either neighbouring bin's value is the right one
    lo, hi = IO.bracket(cdf, mids, u, 1e-12)
    zr = zf_ref.numpy()
    assert ((zr >= lo - 1e-9) & (zr <= hi + 1e-9)).all()
    assert (np.abs(zf - zr) > 1e-9).mean() < 0.01
    assert (np.diff(zf, axis=-1) >= 0).all()
    assert (zf >= mids[:, :1] - 1e-12).all() and (zf <= mids[:, -1:] + 1e-12).all()
    assert cdf.shape == (B, Nc - 1) and np.allclose(cdf[:, -1], 1.0)
    if kind == "zero":                              # uniform pdf over the bins: the fine depths are equally spaced in c
        np.testing.assert_allclose(cdf, np.broadcast_to(np.linspace(0, 1, Nc - 1), cdf.shape), atol=1e-12)


def test_oracle_merge_is_stable_and_sorted():
    z = np.array([[1.0, 2.0, 2.0, 3.0]])
    zf = np.array([[0.5, 2.0, 3.0, 4.0]])
    zm, src = IO.merge(z, zf)
    assert zm.tolist() == [[0.5, 1.0, 2.0, 2.0, 2.0, 3.0, 3.0, 4.0]]
    assert src.tolist() == [[4, 0, 1, 2, 5, 3, 6, 7]]          # coarse before fine on ties


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


def test_native_importance_sample_refuses_bad_arguments(lib):
    fake = 256        # never dereferenced: the arguments are checked before any launch

    def args(**kw):
        a = dict(sigma=fake, z=fake, rays_d=fake, u_table=fake, u_jitter=None, B=16, Nc=64, Nf=128, z_fine=fake,
                 z_merged=fake, merge_src=fake)
        a.update(kw)
        return list(a.values()) + [None]

    for kw, msg in ((dict(Nc=2), "Nc >= 3"), (dict(Nc=-1), "Nc >= 3"), (dict(Nf=0), "Nf >= 1"),
                    (dict(Nc=512, Nf=513), "Nc \\+ Nf <= 1024"), (dict(u_jitter=fake), "exactly one"),
                    (dict(u_table=None), "exactly one"), (dict(B=-1), "negative B")):
        with pytest.raises(ValueError, match=msg):
            lib.call("b2n_importance_sample", *args(**kw))
    for name in ("sigma", "z", "rays_d", "z_fine", "z_merged", "merge_src"):
        with pytest.raises(ValueError, match="null pointer"):
            lib.call("b2n_importance_sample", *args(**{name: None}))
    lib.call("b2n_importance_sample", *args(B=0, sigma=None, z_fine=None))      # empty input: a no-op
    lib.call("b2n_importance_sample", *args(B=0, Nc=1000, Nf=24))


def test_python_entry_points_refuse_bad_arguments(lib):
    import b2n
    model = torch.nn.Identity()
    ro = rd = torch.zeros(4, 3)
    for nc, nf in ((2, 8), (64, 0), (1000, 25), (64.0, 8), (True, 8)):
        with pytest.raises(ValueError, match="n_coarse|n_fine"):
            b2n.render_rays_hierarchical(model, ro, rd, 2.0, 6.0, nc, nf, True)
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.render_rays_hierarchical(model, ro, rd, 2.0, 6.0, 64, 128, True)
    with pytest.raises(ValueError, match="chunk"):
        b2n.render_image_hierarchical(model, torch.zeros(2, 2, 3), torch.zeros(2, 2, 3), 2.0, 6.0, 64, 128, 0, True)
    assert model.training
