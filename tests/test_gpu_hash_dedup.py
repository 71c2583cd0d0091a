"""The warp-level entry merge of the spatially ordered table gradient (b2n_hash_bwd_ordered; b2n_debug_hash_dedup, default
res <= 122): corners by vertex parity, equal entries summed across the warp before the red.global.  Against the fp64
reference of test_gpu_hash_fullsize, per element (|G - G_ref| <= 1e-4 sum |w g|, and with g > 0 exactly the entries a
contribution reaches):

* at C2 size, with every level merged (the shipped window is covered by test_gpu_hash_order);
* warps built to stress the merge, with the shipped window and every level merged: 64 points in one cell, points on
  lattice planes and box faces (weights exactly 0 or 1), zero-gradient samples among live ones and levels no live sample
  reaches, different vertices that hash to one entry in the same slot of one warp, a ragged last warp."""
import pytest
import torch

from _util import record
from test_gpu_hash_fullsize import BOUND, DEV, L, TOL_G, _Env, _reference, _table_check
from test_gpu_hash_order import _bwd_ordered, _order

pytestmark = pytest.mark.gpu
ALL = 1 << 20                     # dedup_res above every level's resolution: every level merged


@pytest.fixture(scope="module")
def env():
    e = _Env()
    yield e
    e.refs.clear()
    torch.cuda.empty_cache()


def test_table_gradient_every_level_merged_at_c2_size(env):
    C = env.C
    x = env.sets["dense"]
    P = x.shape[0]
    (geom, lv, table, G_ref, A), _ = env.reference(19, "dense")
    order, xs = _order(C, x, P)
    G = torch.empty(geom.n_params, device=DEV)
    bad = []
    with C.hash_dedup(ALL):
        for k, g in env.grads("dense").items():
            G.zero_()
            _bwd_ordered(C, xs, order, P, table, geom, g, 2 * L, 0, G)
            r, exact = _table_check(G, G_ref[k], A[k], k == "pos")
            record(f"hash_dedup[dense]:g_table/A[all levels,{k}]", r)
            if not (r <= TOL_G and exact):
                bad.append((k, r, exact))
    assert not bad, bad


def _colliding_cells(lev, gen, n):
    """n pairs of cell corners (x0, y0, z0) != (x1, y1, z1) of a hashed level with the same entry and the same (y, z)
    parity: one parity slot of a warp holds both"""
    from oracle import nerf_oracle as O
    cells = []
    while len(cells) < 2 * n:
        a = torch.randint(1, lev.res - 2, (3,), generator=gen)
        yz = torch.randint(1, lev.res // 2 - 2, (4096, 2), generator=gen) * 2 + (a[1:] & 1)
        e = O.hash_corner_index(lev, a[0:1], a[1:2], a[2:3])
        # x column with the same low bits: x1 = e ^ hash(0, y1, z1) (x carries hash prime 1)
        x1 = e ^ O.hash_corner_index(lev, torch.zeros(4096, dtype=torch.long), yz[:, 0], yz[:, 1])
        ok = (x1 >= 1) & (x1 < lev.res - 2) & ((yz != a[1:]).any(1))
        if ok.any():
            i = int(ok.nonzero()[0])
            b = torch.stack([x1[i], yz[i, 0], yz[i, 1]])
            assert int(O.hash_corner_index(lev, b[0:1], b[1:2], b[2:3])) == int(e)
            cells += [a, b]
    return torch.stack(cells).double()


def _adversarial(case, lv, gen):
    """points (world coordinates) and incoming gradients [P, 2 L] of one case"""
    P = 16 * 4
    grad = 1.0 - torch.rand(P, 2 * L, generator=gen)                     # (0, 1]
    if case == "one_cell":                                               # every point of the warp in one level-8 cell
        lev = lv[8]
        c = torch.randint(2, lev.res - 3, (3,), generator=gen).double()
        u = (c + 0.1 + 0.8 * torch.rand(P, 3, generator=gen, dtype=torch.float64) - 0.5) / lev.scale
    elif case == "faces":
        # x01 = 0.5 is a lattice plane of levels 0-3 (odd integer scales): weight exactly 0 or 1 along that axis; 0 and 1
        # are the box faces
        u = torch.tensor([0.5, 0.0, 1.0], dtype=torch.float64)[torch.randint(0, 3, (P, 3), generator=gen)]
        jitter = 0.45 + 0.1 * torch.rand(P, 3, generator=gen, dtype=torch.float64)
        u = torch.where(torch.rand(P, 3, generator=gen) < 0.3, jitter, u)
    elif case == "zero_grads":
        u = 0.4 + 0.05 * torch.rand(P, 3, generator=gen, dtype=torch.float64)
        grad[torch.rand(P, generator=gen) < 0.5] = 0.0
        grad[:, 6:10] = 0.0                                              # levels 3 and 4: no live sample at all
    elif case == "collisions":                                           # one warp: 8 colliding vertex pairs at level 13
        P = 16
        grad = 1.0 - torch.rand(P, 2 * L, generator=gen)
        u = (_colliding_cells(lv[13], gen, 8) + 0.25) / lv[13].scale
    elif case == "ragged":                                               # 5 warps + 7 points
        P = 16 * 5 + 7
        grad = 1.0 - torch.rand(P, 2 * L, generator=gen)
        u = 0.3 + 0.02 * torch.rand(P, 3, generator=gen, dtype=torch.float64)
    x = (u.clamp(0, 1) * (2 * BOUND) - BOUND).float()
    return x.to(DEV), grad.to(DEV)


@pytest.mark.parametrize("case", ["one_cell", "faces", "zero_grads", "collisions", "ragged"])
def test_adversarial_warps(env, case):
    C = env.C
    geom, lv, table = env.geometry(19)
    x, g = _adversarial(case, lv, torch.Generator().manual_seed(len(case)))
    P = x.shape[0]
    G_ref, A, _ = _reference(x, [table], lv, {"g": g})
    order, xs = _order(C, x, P)
    for d in (-1, ALL):
        G = torch.zeros(geom.n_params, device=DEV)
        with C.hash_dedup(d):
            _bwd_ordered(C, xs, order, P, table, geom, g, 2 * L, 0, G)
        r, exact = _table_check(G, G_ref["g"][0], A["g"][0], True)
        assert record(f"hash_dedup[{case}]:g_table/A[d{d}]", r) <= TOL_G and exact, (d, r, exact)
