"""CPU checks of the fast-render contract: the float64 oracle of _render_oracle.py against the reference compositing of
oracle/nerf_oracle.py at eps = 0, its truncation bound for eps > 0, and the argument checks of the b2n_render_* entry
points, which refuse bad input before any launch."""
import math

import numpy as np
import pytest
import torch

import _render_oracle as RO
from oracle import nerf_oracle as O


def _inputs(B, N, seed, near=2.0, far=6.0):
    rng = np.random.RandomState(seed)
    z = np.linspace(near, far, N)
    sigma = rng.exponential(2.0, (B, N)) * (rng.rand(B, N) < 0.6)
    rgb = rng.rand(B, N, 3)
    d = rng.randn(B, 3)
    return sigma, rgb, z, d


@pytest.mark.parametrize("B,N", [(64, 128), (32, 33), (16, 2), (8, 1)])
def test_oracle_at_eps_zero_equals_volume_render(B, N):
    sigma, rgb, z, d = _inputs(B, N, seed=N)
    bg = np.array([1.0, 0.5, 0.25])
    color, depth, acc, n, _ = RO.render(sigma, rgb, z, np.linalg.norm(d, axis=-1), np.ones((B, N), bool), 0.0, bg)
    t = torch.from_numpy
    zz = t(np.broadcast_to(z, (B, N)).copy())
    rc, rd, ra = O.volume_render(t(rgb), t(sigma), zz, t(d), t(bg))
    np.testing.assert_allclose(color, rc.numpy(), rtol=0, atol=1e-12)
    np.testing.assert_allclose(depth, rd.numpy(), rtol=0, atol=1e-12 * 6.0)
    np.testing.assert_allclose(acc, ra.numpy(), rtol=0, atol=1e-12)
    assert (n == (N if N > 1 else 0)).all()


def test_oracle_inactive_samples_are_skipped():
    """an inactive sample is a sample with sigma = rgb = 0 (what the masked compositor makes of it), up to the 1e-10 of
    its transmittance factor 1 - 0 + 1e-10, which is 1 in fp32 but not in float64"""
    B, N = 32, 64
    sigma, rgb, z, d = _inputs(B, N, seed=5)
    active = np.random.RandomState(6).rand(B, N) < 0.5
    dn = np.linalg.norm(d, axis=-1)
    a = RO.render(sigma, rgb, z, dn, active, 0.0, np.ones(3))
    b = RO.render(sigma * active, rgb * active[..., None], z, dn, np.ones((B, N), bool), 0.0, np.ones(3))
    for x, y in zip(a[:3], b[:3]):
        np.testing.assert_allclose(x, y, rtol=0, atol=N * 1e-10 * 6.0)
    assert (a[3] == active.sum(-1)).all()


@pytest.mark.parametrize("eps", [1e-4, 1e-2, 0.3])
def test_oracle_truncation_bound(eps):
    B, N, far = 256, 128, 6.0
    sigma, rgb, z, d = _inputs(B, N, seed=11, far=far)
    dn = np.linalg.norm(d, axis=-1)
    bg = np.random.RandomState(12).rand(B, 3)
    active = np.ones((B, N), bool)
    full = RO.render(sigma, rgb, z, dn, active, 0.0, bg)
    cut = RO.render(sigma, rgb, z, dn, active, eps, bg)
    assert (cut[3] <= full[3]).all() and (cut[3] < full[3]).any()
    assert np.abs(cut[0] - full[0]).max() <= eps
    assert np.abs(cut[2] - full[2]).max() <= eps
    assert np.abs(cut[1] - full[1]).max() <= eps * far


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


@pytest.mark.parametrize("eps", [-1e-6, 1.0, 2.0, math.nan, math.inf])
def test_native_composite_refuses_bad_threshold(lib, eps):
    fake = 256        # never dereferenced: the arguments are checked before any launch
    with pytest.raises(ValueError, match="b2n_render_composite"):
        lib.call("b2n_render_composite", fake, fake, fake, fake, 16, 8, eps, fake, fake, 4, fake, fake + 64, fake,
                 fake, None)


def test_native_entry_points_refuse_bad_sizes(lib):
    fake = 256
    with pytest.raises(ValueError, match="N <= 1024"):
        lib.call("b2n_render_begin", fake, 16, 1025, fake, fake, fake, fake, None)
    with pytest.raises(ValueError, match="null pointer"):
        lib.call("b2n_render_begin", None, 16, 8, fake, fake, fake, fake, None)
    emit = [fake, fake, None, fake, fake, 16, 8, fake, fake, 4, 2, fake, fake, fake, None, fake, fake, None]
    for i, v in ((10, 9), (10, 0), (9, 17)):         # K > N, K == 0, n_alive > B
        args = list(emit)
        args[i] = v
        with pytest.raises(ValueError, match="b2n_render_emit"):
            lib.call("b2n_render_emit", *args)
    args = list(emit)
    args[14] = fake                                 # t_out without times
    with pytest.raises(ValueError, match="t_out needs times"):
        lib.call("b2n_render_emit", *args)
    with pytest.raises(ValueError, match="alias"):
        lib.call("b2n_render_composite", fake, fake, fake, fake, 16, 8, 0.0, fake, fake, 4, fake, fake, fake, fake,
                 None)
    with pytest.raises(ValueError, match="null pointer"):
        lib.call("b2n_render_finish", fake, 16, None, 0, fake, fake, fake, None)
    assert lib.lib.b2n_render_scratch(1000) >= 4 * (4 * 1000 + 4)
