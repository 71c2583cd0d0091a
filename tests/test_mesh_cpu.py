"""CPU checks of the surface-extraction rules (include/b2nerf.h b2n_mesh_*, DESIGN.md §5f) through their numpy float32
restatement in _mesh_oracle.py: per-tetrahedron cases and winding, closed 2-manifold output with the right topology and
orientation on small fields, the empty and full fields, and the PLY writer."""
import numpy as np
import pytest
import torch

import _mesh_oracle as M

EDGES = [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]


def _axis(R, bound=1.0):
    return torch.linspace(-bound, bound, R)


@pytest.mark.parametrize("odd", [0, 1])
@pytest.mark.parametrize("case", range(16))
def test_single_tetrahedron_case_and_winding(case, odd):
    """Each of the 16 inside/outside patterns of one tetrahedron, positively and negatively oriented: the number of
    triangles (0, 1 or 2), that they cover exactly the crossing edges, and that every normal points from the inside
    corners to the outside ones.  The complementary pattern (inside and outside swapped) gives the same triangles with
    the opposite winding."""
    perm = M.PERMS[1] if odd else M.PERMS[0]
    assert M.parity(perm) == odd
    lv = np.array(M.tet_corners(perm), float)
    vol = np.linalg.det(np.stack([lv[1] - lv[0], lv[2] - lv[0], lv[3] - lv[0]]))
    assert np.sign(vol) == (-1 if odd else 1)
    n_in = bin(case).count("1")
    tris = M.tet_triangles(case, odd)
    assert len(tris) == {0: 0, 1: 1, 2: 2, 3: 1, 4: 0}[n_in]
    crossing = {(m, n) for (m, n) in EDGES if (case >> m & 1) != (case >> n & 1)}
    assert {e for t in tris for e in t} == crossing
    rng = np.random.default_rng(case)
    for _ in range(4):                                  # any position along the edges: the winding is combinatorial
        tpos = {e: rng.uniform(0.05, 0.95) for e in EDGES}
        pos = {e: lv[e[0]] + tpos[e] * (lv[e[1]] - lv[e[0]]) for e in EDGES}
        for t in tris:
            a, b, c = (pos[e] for e in t)
            nrm = np.cross(b - a, c - a)
            for m in range(4):
                side = np.dot(nrm, lv[m] - a)
                if abs(side) < 1e-12:
                    continue                            # a corner in the triangle's plane (the quad's own corners)
                assert (side < 0) == bool(case >> m & 1), (case, odd, t, m)
    comp = M.tet_triangles(15 - case, odd)
    assert sorted(tuple(sorted(t)) for t in comp) == sorted(tuple(sorted(t)) for t in tris)
    for t in tris:                                      # reversed cyclic order
        u = next(u for u in comp if set(u) == set(t))
        assert any(u == (t[k], t[(k + 2) % 3], t[(k + 1) % 3]) for k in range(3)), (t, u)


@pytest.mark.parametrize("name,R", [("ball", 17), ("ball", 24), ("torus", 28), ("two_balls", 26), ("slab", 12)])
def test_oracle_mesh_is_closed_oriented_manifold(name, R):
    ax = _axis(R)
    verts, faces = M.extract(M.field(name, ax).numpy(), M.TAU, ax.numpy())
    assert M.euler(verts, faces) == M.EULER[name]
    assert M.signed_volume(verts, faces) > 0
    h = float(ax[1] - ax[0])
    if name in M.ANALYTIC_VOLUME:
        assert abs(M.signed_volume(verts, faces) - M.ANALYTIC_VOLUME[name]) < M.ANALYTIC_AREA[name] * h


def test_oracle_noise_field_is_manifold():
    ax = _axis(9)
    verts, faces = M.extract(M.field("noise", ax).numpy(), M.TAU, ax.numpy())
    M.check_closed_manifold(verts, faces)
    assert M.signed_volume(verts, faces) > 0


def test_oracle_empty_field_gives_empty_mesh():
    ax = _axis(6)
    verts, faces = M.extract(M.field("empty", ax).numpy(), M.TAU, ax.numpy())
    assert verts.shape == (0, 3) and faces.shape == (0, 3)


@pytest.mark.parametrize("R", [2, 5])
def test_oracle_full_field_gives_closed_box(R):
    """every point inside: the surface closes around the whole lattice on the box half a spacing outside it
    (sigma = 2 tau against the sigma = 0 ring puts every vertex half-way).  Piecewise-linear interpolation chamfers
    the box edges that do not run along the main diagonal, so the volume lies between the lattice's box and that box."""
    bound = 1.25
    ax = _axis(R, bound)
    verts, faces = M.extract(M.field("full", ax).numpy(), M.TAU, ax.numpy())
    assert M.euler(verts, faces) == 2
    h = float(ax[1] - ax[0])
    half = bound + h / 2
    assert np.allclose(np.abs(verts).max(axis=1), half, atol=1e-6)
    assert np.allclose(verts.min(axis=0), -half, atol=1e-6) and np.allclose(verts.max(axis=0), half, atol=1e-6)
    assert (2 * bound) ** 3 < M.signed_volume(verts, faces) < (2 * half) ** 3


def test_oracle_vertices_follow_the_float32_rule():
    """a vertex is p + t (q - p) with t = (tau - sigma_p) / (sigma_q - sigma_p), evaluated in float32 step by step"""
    ax = _axis(3, 0.7)
    sig = np.zeros((3, 3, 3), np.float32)
    sig[1, 1, 1] = 1.7
    verts, faces = M.extract(sig, 0.3, ax.numpy())
    assert len(verts) == 14 and len(faces) == 24         # the 14 lattice edges around the single inside point
    ext = M.extended_axis(ax.numpy())
    # the inside point is (2,2,2) of the padded lattice; the lowest point with a crossing edge is (1,1,1), along xyz
    t =(np.float32(0.3) - np.float32(0.0)) / (np.float32(1.7) - np.float32(0.0))
    want = ext[1] + t * (ext[2] - ext[1])
    assert verts.dtype == np.float32 and np.array_equal(verts[0], np.full(3, want, np.float32))


def test_write_ply_round_trip(tmp_path):
    import __graft_entry__ as ge
    ge.build()
    from b2n.mesh import write_ply
    ax = _axis(10)
    verts, faces = M.extract(M.field("ball", ax).numpy(), M.TAU, ax.numpy())
    path = tmp_path / "ball.ply"
    write_ply(str(path), torch.from_numpy(verts), torch.from_numpy(faces))
    raw = path.read_bytes()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    header = raw[:end].decode("ascii").splitlines()
    assert header[:2] == ["ply", "format binary_little_endian 1.0"]
    assert f"element vertex {len(verts)}" in header and f"element face {len(faces)}" in header
    body = raw[end:]
    v = np.frombuffer(body[:12 * len(verts)], "<f4").reshape(-1, 3)
    rec = np.frombuffer(body[12 * len(verts):], dtype=[("n", "u1"), ("v", "<i4", (3,))])
    assert np.array_equal(v, verts) and (rec["n"] == 3).all() and np.array_equal(rec["v"], faces)
