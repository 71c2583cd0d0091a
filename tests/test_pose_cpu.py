"""CPU checks of the pose-refinement contract: the float64 oracle of _pose_oracle.py against scipy's rotation vector
and central differences, the Rodrigues map of b2n/pose.py (exact I at omega = 0, continuous across its Taylor
threshold, a finite gradient at 0), and the argument checks of the native and the Python layer, which refuse bad input
before any launch."""
import math

import numpy as np
import pytest
import torch
from scipy.spatial.transform import Rotation

import _pose_oracle as PO

H, W, FOCAL = 12, 10, 11.5


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


def _omegas(n, seed=0):
    rng = np.random.RandomState(seed)
    axis = rng.randn(n, 3)
    axis /= np.linalg.norm(axis, axis=1, keepdims=True)
    ang = np.concatenate([[0.0, 1e-9, 1e-7, 1e-6, 1e-3, 0.03, 0.5, 2.0, 3.1], rng.uniform(0, 3, n - 9)])
    return torch.from_numpy(axis * ang[:, None])


def _poses(V, seed=0):
    rng = np.random.RandomState(seed)
    R = Rotation.random(V, random_state=rng).as_matrix()
    P = np.zeros((V, 4, 4))
    P[:, :3, :3], P[:, :3, 3], P[:, 3, 3] = R, rng.randn(V, 3) * 3, 1.0
    return torch.from_numpy(P).float()


def test_oracle_rodrigues_is_scipys_rotation_vector():
    w = _omegas(40)
    np.testing.assert_allclose(PO.exp_so3(w).numpy(), Rotation.from_rotvec(w.numpy()).as_matrix(), rtol=0, atol=2e-15)


def test_product_rodrigues_matches_scipy_and_is_exact_at_zero(lib):
    from b2n import pose
    w = _omegas(40, seed=1)
    np.testing.assert_allclose(pose.so3_exp(w).numpy(), Rotation.from_rotvec(w.numpy()).as_matrix(), rtol=0, atol=3e-15)
    assert torch.equal(pose.so3_exp(torch.zeros(5, 3)), torch.eye(3).expand(5, 3, 3))
    P = _poses(7)
    assert torch.equal(pose.compose(P, torch.zeros(7, 6)), P)             # c2w' is c2w, bit for bit, at xi = 0
    xi = torch.from_numpy(np.random.RandomState(2).randn(7, 6) * 0.1)
    np.testing.assert_allclose(pose.compose(P.double(), xi).numpy(), PO.corrected(P, xi).numpy(), rtol=0, atol=1e-14)


def test_taylor_branch_is_continuous_with_a_finite_gradient_at_zero(lib):
    from b2n import pose
    axis = torch.tensor([0.3, -0.5, 0.8], dtype=torch.float64)
    axis = axis / axis.norm()
    thr = math.sqrt(pose.TAYLOR_THETA2)
    # both sides of the threshold: the map's step there is the exact map's step (|dR/dtheta| * 2e-9 * theta)
    ts = (thr * (1 - 1e-9), thr * (1 + 1e-9))
    got = [pose.so3_exp(axis * t) for t in ts]
    ref = [torch.from_numpy(Rotation.from_rotvec((axis * t).numpy()).as_matrix()) for t in ts]
    for a, b in zip(got, ref):
        assert float((a - b).abs().max()) < 1e-15
    assert float(((got[1] - got[0]) - (ref[1] - ref[0])).abs().max()) < 1e-15
    # at 0 (step 1 of every run) the gradient is finite and equals d/domega of sum(G * exp(omega)) = vee(G - G^T)
    G = torch.from_numpy(np.random.RandomState(3).randn(3, 3))
    for dtype in (torch.float32, torch.float64):
        w = torch.zeros(3, dtype=dtype, requires_grad=True)
        (g,) = torch.autograd.grad((pose.so3_exp(w) * G.to(dtype)).sum(), w)
        assert torch.isfinite(g).all()
        A = G - G.T
        np.testing.assert_allclose(g.double().numpy(), [A[2, 1], A[0, 2], A[1, 0]], rtol=1e-6)
    # the oracle's gradient at 0 too
    w = torch.zeros(1, 3, dtype=torch.float64, requires_grad=True)
    (g,) = torch.autograd.grad((PO.exp_so3(w)[0] * G).sum(), w)
    assert torch.isfinite(g).all()


def test_oracle_gradient_matches_central_differences():
    V, B, N = 3, 9, 5
    rng = np.random.RandomState(4)
    P = _poses(V, seed=5)
    picks = (torch.from_numpy(rng.randint(0, V, B)), torch.from_numpy(rng.randint(0, H, B)),
             torch.from_numpy(rng.randint(0, W, B)))
    z = torch.from_numpy(np.sort(rng.uniform(2, 6, (B, N)), 1))
    g_pts = torch.from_numpy(rng.randn(B, N, 3))
    xi0 = torch.from_numpy(rng.randn(V, 6) * 0.05)
    xi0[0] = 0.0                                                          # one view at xi = 0

    def L(x):
        o, d = PO.rays(PO.corrected(P, x), *picks, H, W, FOCAL, 0.7)
        return float((PO.points(o, d, z) * g_pts).sum())

    g = PO.xi_grad(P, xi0, picks, H, W, FOCAL, 0.7, z, g_pts)
    h = 1e-6
    for v in range(V):
        for k in range(6):
            xp, xm = xi0.clone(), xi0.clone()
            xp[v, k] += h
            xm[v, k] -= h
            fd = (L(xp) - L(xm)) / (2 * h)
            assert math.isclose(float(g[v, k]), fd, rel_tol=1e-6, abs_tol=1e-7), (v, k, float(g[v, k]), fd)
    # the two-stage form (points -> rays -> poses) is the same gradient: the one the kernels compute
    o, d = PO.rays(PO.corrected(P, xi0), *picks, H, W, FOCAL, 0.7)
    g_o, g_d = PO.points_bwd(z, g_pts)
    gP = PO.rays_bwd(PO.corrected(P, xi0), *picks, H, W, FOCAL, 0.7, g_o, g_d)
    x = xi0.clone().requires_grad_(True)
    (g2,) = torch.autograd.grad((PO.corrected(P, x) * gP).sum(), x)
    np.testing.assert_allclose(g2.numpy(), g.numpy(), rtol=1e-10, atol=1e-12)


def test_oracle_direction_gradient_has_no_component_along_the_ray():
    """the normalisation Jacobian (I - dh dh^T)/|d| removes any component along dh: the |d| terms of the composite
    and the distortion loss would contribute exactly zero, which is why they need no ray gradient"""
    P = _poses(2, seed=6)
    picks = (torch.tensor([0, 1, 1]), torch.tensor([3, 0, 11]), torch.tensor([9, 4, 0]))
    o, d = PO.rays(P.double(), *picks, H, W, FOCAL, 1.0)
    g = PO.rays_bwd(P, *picks, H, W, FOCAL, 1.0, torch.zeros(3, 3), d * torch.tensor([[2.0], [-1.0], [0.5]]))
    assert float(g.abs().max()) < 1e-14


@pytest.mark.parametrize("entry", ["b2n_march_points_bwd", "b2n_sample_rays_bwd"])
def test_native_entry_points_refuse_bad_arguments(lib, entry):
    p = 64                                                                # a non-null pointer, never dereferenced
    if entry == "b2n_march_points_bwd":
        bad = [((p, None, None, p, 4, 0, p, p, None), "bad B or N"),
               ((p, None, None, p, 4, 4097, p, p, None), "bad B or N"),
               ((p, None, None, p, -1, 8, p, p, None), "bad B or N"),
               ((None, None, None, p, 4, 8, p, p, None), "null pointer"),
               ((p, None, None, p, 4, 8, None, p, None), "null pointer"),
               ((p, p, None, p, 4, 8, p, p, None), "ray_offset"),
               ((p, None, None, p, 2 ** 28, 8, p, p, None), "int32")]
        lib.call(entry, None, None, None, None, 0, 8, None, None, None)      # B = 0: a no-op
    else:
        ok = [p, p, p, p, 4, 3, H, W, FOCAL, 1.0, p, p, p, p, None]

        def with_(**kw):
            a = list(ok)
            for k, v in kw.items():
                a[int(k[1:])] = v
            return tuple(a)
        bad = [(with_(a5=0), "bad shape"), (with_(a4=-1), "bad shape"), (with_(a4=2 ** 31), "bad shape"),
               (with_(a6=0), "bad shape"), (with_(a7=0), "bad shape"), (with_(a8=0.0), "bad shape"),
               (with_(a0=None), "null pointer"), (with_(a12=None), "null pointer"), (with_(a13=None), "null pointer"),
               (with_(a11=None), "null pointer"), (with_(a1=None), "null pointer")]
        assert lib.lib.b2n_sample_rays_bwd_scratch(-1, 3) == 0 and lib.lib.b2n_sample_rays_bwd_scratch(4, 0) == 0
    for args, msg in bad:
        with pytest.raises(ValueError, match=msg):
            lib.call(entry, *args)


def test_python_layer_refuses_bad_arguments(lib):
    import b2n
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.PoseRefinement(4, device="cpu")
    for bad in (0, -1, 2.0, True):
        with pytest.raises(ValueError, match="n_views"):
            b2n.PoseRefinement(bad, device="cpu")
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.march.march(torch.zeros(2, 3, requires_grad=True), torch.ones(2, 3), 2.0, 6.0, 8, None)
