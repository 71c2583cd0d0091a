"""GPU tests of surface extraction (b2n.mesh, b2n_mesh_* of include/b2nerf.h): the kernels against the numpy float32
oracle of _mesh_oracle.py (faces equal, vertices bitwise), determinism, the mesh checks at R = 512, the lattice sweep of
a model against DensityGrid.update / NeuralField.density, and the refusals."""
import pytest
import torch

import _mesh_oracle as M

pytestmark = pytest.mark.gpu
DEV = "cuda"
FIELDS = ["ball", "torus", "two_balls", "slab", "empty", "full", "noise"]


@pytest.fixture(scope="module")
def mesh():
    import b2n
    return b2n.mesh


def _lattice(mesh, name, R, bound=1.0):
    ax = mesh.lattice_axis(R, bound, DEV)
    return M.field(name, ax.cpu()).to(DEV).contiguous(), ax.cpu()


def _bits(v):
    return v.contiguous().view(torch.int32)


@pytest.mark.parametrize("R", [2, 33, 64])
@pytest.mark.parametrize("name", FIELDS)
def test_extract_equals_oracle(mesh, name, R):
    sigma, ax = _lattice(mesh, name, R)
    verts, faces = mesh.extract(sigma, M.TAU, 1.0)
    ov, of = M.extract(sigma.cpu().numpy(), M.TAU, ax.numpy())
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32
    assert verts.shape == (len(ov), 3) and faces.shape == (len(of), 3)
    assert torch.equal(faces.cpu(), torch.from_numpy(of))
    assert torch.equal(_bits(verts.cpu()), _bits(torch.from_numpy(ov)))
    verts2, faces2 = mesh.extract(sigma, M.TAU, 1.0)
    assert torch.equal(_bits(verts2), _bits(verts)) and torch.equal(faces2, faces)
    if name in M.EULER and R > 2:
        assert M.euler(verts, faces) == M.EULER[name]


@pytest.mark.parametrize("name", ["ball", "torus", "two_balls"])
def test_extract_at_512_against_analytic_surface(mesh, name):
    R, bound = 512, 1.0
    ax = mesh.lattice_axis(R, bound, DEV)
    x, y, z = M.grid_points(ax.double())
    sigma = (M.TAU + 4.0 * M.sdf(name, x, y, z)).float().contiguous()
    del x, y, z
    verts, faces = mesh.extract(sigma, M.TAU, bound)
    assert faces.shape[0] > 10 ** 5
    assert M.euler(verts, faces) == M.EULER[name]
    h = float(ax[1] - ax[0])
    v = verts.double()
    dist = M.sdf(name, v[:, 0], v[:, 1], v[:, 2]).abs()
    assert float(dist.max()) <= h
    vol = M.signed_volume(verts, faces)
    assert abs(vol - M.ANALYTIC_VOLUME[name]) <= M.ANALYTIC_AREA[name] * h


def _part2_model():
    from src.core import NeuralField
    torch.manual_seed(0)
    return NeuralField(dict(mode="part2_instant", scene_bound=1.5)).to(DEV)


def test_density_lattice_equals_density_grid_update(mesh):
    from src.renderer import DensityGrid
    model = _part2_model().eval()
    sigma = mesh.density_lattice(model, 128, 1.5)
    grid = DensityGrid(resolution=128, bound=1.5, threshold=0.01).to(DEV)
    grid.update(model, device=DEV)
    assert sigma.shape == (128, 128, 128) and torch.equal(_bits(sigma), _bits(grid.grid))


def test_density_lattice_part4_equals_model_density(mesh):
    from src.core import NeuralField
    torch.manual_seed(1)
    model = NeuralField(dict(mode="part4", scene_bound=1.5, log2_hashmap_size=16, deform_n_levels=12,
                             deform_log2_hashmap_size=14)).to(DEV).eval()
    R = 48
    sigma = mesh.density_lattice(model, R, 1.5, t=0.5)
    ax = mesh.lattice_axis(R, 1.5, DEV)
    pts = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), -1).reshape(-1, 3).contiguous()
    with torch.no_grad():
        ref = model.density(pts, t=torch.full((pts.shape[0], 1), 0.5, device=DEV))
    assert torch.equal(_bits(sigma.reshape(-1)), _bits(ref.reshape(-1)))


def test_density_lattice_restores_training_mode(mesh):
    model = _part2_model()
    model.train()
    mesh.density_lattice(model, 16, 1.5)
    assert model.training
    model.eval()
    mesh.density_lattice(model, 16, 1.5)
    assert not model.training


def test_density_lattice_without_density_method(mesh):
    """a model without ``density`` is called with zero view directions, like DensityGrid.update calls it"""
    model = _part2_model().eval()

    class NoDensity(torch.nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m = m

        def forward(self, *a, **k):
            return self.m(*a, **k)
    a = mesh.density_lattice(model, 40, 1.5)
    b = mesh.density_lattice(NoDensity(model), 40, 1.5)
    assert torch.equal(_bits(a), _bits(b))


def test_extract_mesh_equals_extract_of_density_lattice(mesh):
    model = _part2_model().eval()
    sigma = mesh.density_lattice(model, 64, 1.5)
    thr = max(float(sigma.flatten().quantile(0.7)), 1e-6)
    v1, f1 = mesh.extract_mesh(model, 64, thr, 1.5)
    v2, f2 = mesh.extract(sigma, thr, 1.5)
    assert f1.shape[0] > 0
    assert torch.equal(_bits(v1), _bits(v2)) and torch.equal(f1, f2)
    M.check_closed_manifold(v1, f1)


def test_refusals_before_any_launch(mesh):
    from b2n import _lib
    good = torch.ones(4, 4, 4, device=DEV)
    bad = [
        (torch.ones(1, 1, 1, device=DEV), 0.5),                      # R < 2
        (torch.empty(1025, 1025, 1025, device=DEV), 0.5),            # R > 1024
        (good, 0.0), (good, -1.0), (good, float("nan")), (good, float("inf")),
        (good.cpu(), 0.5),
        (good.transpose(0, 1), 0.5),
        (torch.ones(4, 4, 5, device=DEV), 0.5), (torch.ones(4, 16, device=DEV), 0.5),
        (good.double(), 0.5),
    ]
    model = _part2_model()
    torch.cuda.synchronize()
    n0 = _lib.LAUNCHES["count"]
    for sigma, tau in bad:
        with pytest.raises(ValueError):
            mesh.extract(sigma, tau, 1.0)
    del bad
    for R in (1, 1025):
        with pytest.raises(ValueError):
            mesh.density_lattice(model, R, 1.5)
    assert _lib.LAUNCHES["count"] == n0
    # the C entry points refuse on their own (argument checks precede every launch)
    scratch = torch.empty(_lib.lib.b2n_mesh_scratch(4), device=DEV, dtype=torch.uint8)
    totals = torch.empty(2, device=DEV, dtype=torch.int64)
    assert _lib.lib.b2n_mesh_scratch(1) == 0 and _lib.lib.b2n_mesh_scratch(1025) == 0
    for R, tau in ((1, 0.5), (1025, 0.5), (4, 0.0), (4, -2.0)):
        with pytest.raises(ValueError, match="b2n_mesh_count"):
            _lib.call("b2n_mesh_count", _lib.ptr(good), R, tau, _lib.ptr(scratch), _lib.ptr(totals), _lib.stream())
    ext = torch.zeros(6, device=DEV)
    out = torch.empty(8, 3, device=DEV)
    for V, F in ((2 ** 31, 8), (8, 2 ** 31), (-1, 0)):
        with pytest.raises(ValueError, match="b2n_mesh_emit"):
            _lib.call("b2n_mesh_emit", _lib.ptr(good), _lib.ptr(ext), 4, 0.5, _lib.ptr(scratch), V, F, _lib.ptr(out),
                      _lib.ptr(out), _lib.stream())


def test_overflow_refused_on_large_noise_field(mesh):
    """i.i.d. noise around tau at R = 1024: about 3.5 crossing edges per point, so V passes 2^31; the totals are exact
    int64 and extract refuses instead of wrapping"""
    R = 1024
    g = torch.Generator(device=DEV).manual_seed(5)
    sigma = torch.rand(R, R, R, device=DEV, generator=g) + 0.5
    with pytest.raises(ValueError, match="2\\^31"):
        mesh.extract(sigma, 1.0, 1.0)
    del sigma
    torch.cuda.empty_cache()
