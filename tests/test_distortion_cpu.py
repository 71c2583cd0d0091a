"""CPU checks of the distortion-loss contract: the float64 double-sum oracle of _distortion_oracle.py against the O(N)
prefix-sum form and its closed-form dL/dw that the kernels use, hand cases, central finite differences of the sigma
gradient, and the argument checks of b2n_distortion_* and b2n.distortion, which refuse bad input before any launch."""
import math

import pytest
import torch

import _distortion_oracle as DO

NEAR, FAR = 2.0, 6.0


def _rays(B, N, seed, p_active=0.7, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    t = torch.linspace(0.0, 1.0, N, dtype=torch.float64)
    z = NEAR * (1 - t) + FAR * t
    if N > 1:
        mids = 0.5 * (z[1:] + z[:-1])
        lo, hi = torch.cat([z[:1], mids]), torch.cat([mids, z[-1:]])
        z = lo + (hi - lo) * torch.rand(B, N, generator=g, dtype=torch.float64)      # jittered strata: sorted per ray
    else:
        z = NEAR + (FAR - NEAR) * torch.rand(B, 1, generator=g, dtype=torch.float64)
    d = torch.randn(B, 3, generator=g, dtype=torch.float64)
    sigma = torch.empty(B, N, dtype=torch.float64).exponential_(1.0 / scale, generator=g)
    sigma = sigma * (torch.rand(B, N, generator=g, dtype=torch.float64) < p_active)
    return sigma, z.contiguous(), d


@pytest.mark.parametrize("N", [1, 2, 3, 65, 128])
def test_prefix_form_and_grad_w_equal_the_double_sum(N):
    sigma, z, d = _rays(24, N, seed=N)
    w = DO.weights(sigma, z, d.norm(dim=-1))
    mid, width = DO.intervals(z, NEAR, FAR)
    assert (mid[:, 1:] >= mid[:, :-1]).all() and (width >= 0).all()
    L = DO.loss_of_weights(w, mid, width)
    torch.testing.assert_close(DO.prefix_form(w, mid, width), L, rtol=1e-12, atol=1e-15)
    wr = w.detach().clone().requires_grad_(True)
    gw, = torch.autograd.grad(DO.loss_of_weights(wr, mid, width).sum(), wr)
    torch.testing.assert_close(DO.grad_w(w, mid, width), gw, rtol=1e-12, atol=1e-14)
    assert torch.equal(DO.loss(sigma, z, d, NEAR, FAR), L)


def test_hand_cases():
    z = torch.tensor([[2.0, 3.0, 4.0, 5.0]], dtype=torch.float64)
    d = torch.tensor([[0.0, 0.0, 1.0]], dtype=torch.float64)
    mid, width = DO.intervals(z, NEAR, FAR)
    torch.testing.assert_close(mid, torch.tensor([[0.125, 0.375, 0.625, 0.875]], dtype=torch.float64))
    torch.testing.assert_close(width, torch.full((1, 4), 0.25, dtype=torch.float64))
    # all weight on one sample: L = w^2 d / 3
    for k in range(4):
        w = torch.zeros(1, 4, dtype=torch.float64)
        w[0, k] = 0.7
        torch.testing.assert_close(DO.loss_of_weights(w, mid, width), torch.tensor([0.49 * 0.25 / 3], dtype=torch.float64))
        torch.testing.assert_close(DO.prefix_form(w, mid, width), torch.tensor([0.49 * 0.25 / 3], dtype=torch.float64))
    # an opaque sample: the weights are one-hot, and so is the loss
    s = torch.tensor([[0.0, 1e4, 0.0, 0.0]], dtype=torch.float64)
    w = DO.weights(s, z, d.norm(dim=-1))
    torch.testing.assert_close(w, torch.tensor([[0.0, 1.0, 0.0, 0.0]], dtype=torch.float64), atol=1e-9, rtol=0)
    torch.testing.assert_close(DO.loss(s, z, d, NEAR, FAR), torch.tensor([0.25 / 3], dtype=torch.float64), atol=1e-9, rtol=0)
    # sigma = 0: no weight, no loss, no gradient
    L, g = DO.loss_and_grad(torch.zeros(3, 4, dtype=torch.float64), z.expand(3, 4), d.expand(3, 3), NEAR, FAR)
    assert torch.equal(L, torch.zeros(3, dtype=torch.float64)) and torch.equal(g, torch.zeros(3, 4, dtype=torch.float64))
    # two equal spikes: 2 w^2 |dm| + 1/3 sum w^2 d
    w = torch.tensor([[0.0, 0.4, 0.0, 0.4]], dtype=torch.float64)
    want = 2 * 0.16 * 0.5 + (0.16 * 0.25 * 2) / 3
    torch.testing.assert_close(DO.loss_of_weights(w, mid, width), torch.tensor([want], dtype=torch.float64))
    torch.testing.assert_close(DO.prefix_form(w, mid, width), torch.tensor([want], dtype=torch.float64))
    # the last interval ends at far, whatever the last compositing delta (1e10)
    z1 = torch.tensor([[3.0]], dtype=torch.float64)
    m1, w1 = DO.intervals(z1, NEAR, FAR)
    assert float(m1) == 0.625 and float(w1) == 0.75


@pytest.mark.parametrize("N", [1, 2, 3, 17])
def test_sigma_gradient_equals_central_differences(N):
    sigma, z, d = _rays(6, N, seed=100 + N, p_active=1.0, scale=0.5)
    sigma = sigma + 0.05                                  # away from sigma = 0 (the last sample's 1e10 interval)
    g_loss = torch.linspace(0.5, 2.0, 6, dtype=torch.float64)
    _, g = DO.loss_and_grad(sigma, z, d, NEAR, FAR, g_loss)
    h = 1e-6
    for r in range(6):
        for i in range(N):
            sp, sm = sigma.clone(), sigma.clone()
            sp[r, i] += h
            sm[r, i] -= h
            fd = float(((DO.loss(sp, z, d, NEAR, FAR) - DO.loss(sm, z, d, NEAR, FAR)) * g_loss).sum()) / (2 * h)
            assert math.isclose(float(g[r, i]), fd, rel_tol=1e-5, abs_tol=1e-9), (r, i, float(g[r, i]), fd)


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


@pytest.mark.parametrize("entry", ["b2n_distortion_fwd", "b2n_distortion_bwd"])
def test_native_entry_points_refuse_bad_arguments(lib, entry):
    fake = 256        # never dereferenced: the arguments are checked before any launch
    bwd = entry.endswith("bwd")

    def args(**kw):
        a = dict(sigma=fake, z=fake, rays_d=fake, mask_words=None, ray_offset=None, B=16, N=64, near=NEAR, far=FAR)
        a.update({k: v for k, v in kw.items() if k in a})
        out = dict(g_loss=fake, g_sigma=fake) if bwd else dict(loss=fake)
        out.update({k: v for k, v in kw.items() if k in out})
        return list(a.values()) + list(out.values()) + [None]

    for kw, msg in ((dict(N=0), "1 <= N <= 1024"), (dict(N=1025), "1 <= N <= 1024"), (dict(N=-3), "1 <= N"),
                    (dict(B=-1), "negative B"), (dict(far=NEAR), "near < far"), (dict(far=1.0), "near < far"),
                    (dict(near=math.nan), "finite"), (dict(far=math.inf), "finite"), (dict(near=-math.inf), "finite"),
                    (dict(near=-3e38, far=3e38), "finite"), (dict(mask_words=fake), "mask_words and ray_offset"),
                    (dict(ray_offset=fake), "mask_words and ray_offset")):
        with pytest.raises(ValueError, match=entry):
            lib.call(entry, *args(**kw))
        with pytest.raises(ValueError, match=msg):
            lib.call(entry, *args(**kw))
    for name in ("sigma", "z", "rays_d") + (("g_loss", "g_sigma") if bwd else ("loss",)):
        with pytest.raises(ValueError, match="null pointer"):
            lib.call(entry, *args(**{name: None}))
    lib.call(entry, *args(B=0, sigma=None, z=None))                  # empty input: a no-op
    with pytest.raises(ValueError, match="1 <= N"):                   # ... but its sizes are still checked
        lib.call(entry, *args(B=0, N=2000))


def test_python_op_refuses_bad_arguments(lib):
    import b2n
    B, N = 4, 40
    s, z, d = torch.zeros(B * N), torch.zeros(B, N), torch.zeros(B, 3)
    mw, off = torch.zeros(B, 2, dtype=torch.int32), torch.zeros(B + 1, dtype=torch.int32)
    for near, far in ((2.0, 2.0), (6.0, 2.0), (math.nan, 6.0), (2.0, math.inf)):
        with pytest.raises(ValueError, match="near and far"):
            b2n.distortion(s, z, d, near, far)
    with pytest.raises(ValueError, match="z must be"):
        b2n.distortion(s, z.reshape(-1), d, NEAR, FAR)
    with pytest.raises(ValueError, match="N <= 1024"):
        b2n.distortion(torch.zeros(1025), torch.zeros(1, 1025), torch.zeros(1, 3), NEAR, FAR)
    with pytest.raises(ValueError, match="rays_d"):
        b2n.distortion(s, z, torch.zeros(B + 1, 3), NEAR, FAR)
    with pytest.raises(ValueError, match="B\\*N"):
        b2n.distortion(torch.zeros(B * N - 1), z, d, NEAR, FAR)
    with pytest.raises(ValueError, match="both mask_words and ray_offset"):
        b2n.distortion(s, z, d, NEAR, FAR, mask_words=mw)
    with pytest.raises(ValueError, match="int32"):
        b2n.distortion(s, z, d, NEAR, FAR, mask_words=mw.long(), ray_offset=off)
    with pytest.raises(ValueError, match="mask_words \\[B, 2\\]"):
        b2n.distortion(s, z, d, NEAR, FAR, mask_words=mw[:, :1], ray_offset=off)
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.distortion(s, z, d, NEAR, FAR)
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.distortion(torch.zeros(7), z, d, NEAR, FAR, mask_words=mw, ray_offset=off)
    model = torch.nn.Identity()
    model.mode = "part2_instant"
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.render_rays_distortion(model, torch.zeros(B, 3), torch.ones(B, 3), NEAR, FAR, N, True)
