"""Hash-grid encoder at training size against an fp64 reference (-m gpu).

The sample sets are the C2 step's own: 2^18 rays x 128 jittered samples (near / far 2 / 6) marched by b2n.march through
  dense   an all-ones 128^3 grid (about 24 M points, ray order: runs of samples that share a cell),
  ball    the ball occupancy bench.py uses (short runs, rays that end mid-warp; the row count is kept off every multiple
          of 16 for the static-capacity case),
  morton  the dense set sorted by a 30-bit Morton key (runs far longer than a warp, many crossing warp boundaries).
Every configuration of the F = 2 kernels (b2n_debug_hash_variant 0..3, run-merging threshold 0 .. 200) is compared with
one fp64 evaluation of the same operation, element by element and row by row:

  features  |y - y_ref| <= 2e-6 sum_k |w_k T_e|          eight fp32 products and adds: about 10 ulp
  g_table   |G - G_ref| <= 1e-4 A_e,  A_e = sum |w g|     per table element; with g > 0 also G_e == 0 <=> A_e == 0
  g_x       |g_x - ref| <= 1e-5 sum of |level terms|      per row and coordinate

A max-norm over the whole table is dominated by the coarse levels; a per-element bar makes a run sum that lands on the
wrong entry of a fine level visible.

Measured on a B200 (1000 W power limit): worst g_table / A 1.0e-5 in the shipped configuration (3, 128), 3.6e-5 with
merging off (merge_res 0).  Both are the fp32 rounding of the coarse entries' sums with a positive g, which grows like
sqrt(n) 2^-24 in the n red.global.add an entry receives: about 10^5 per level-0 entry unmerged, up to 8 times fewer
after the warp merge (sqrt(8) = 2.8, the measured ratio is 3.3).  The 1e-4 bar has a margin of about 3 there.

The cell decisions (x01, floor, fractional weights) are made in fp32 exactly as to_unit / locate (b2n_hash.cuh) make them:
in fp64 the reference would put points on a cell boundary into the other cell.  test_cell_decisions_match_oracle pins
these decisions to the CPU oracle's fp32 arithmetic.  Everything after them is float64."""
import math

import pytest
import torch

from _util import record

pytestmark = pytest.mark.gpu
DEV = "cuda"
BOUND = 1.5
L, F = 16, 2
CHUNK = 2 ** 21                     # points per reference chunk: bounded memory at 24 M points
SHIPPED = (3, 128)                  # b2n_encode.cu: g_hash_variant, g_merge_res
# variants 0 / 1 scatter with k_hash_bwd_table(_dense), which ignores the merge threshold
CONFIGS = [(0, 128), (1, 128)] + [(v, m) for v in (2, 3) for m in (0, 24, 64, 128, 200)]
TOL_Y, TOL_G, TOL_X = 2e-6, 1e-4, 1e-5
SEEDS = {"dense": 11, "ball": 12, "morton": 13}


# ------------------------------------------------------------------ fp32 decisions, fp64 arithmetic
def _x01(x):
    """to_unit: clamp((x + b) / (2 b), 0, 1) and the closed-interval mask of the clamp's gradient.  The divisor is a
    tensor: torch evaluates x / python_scalar on CUDA as x * (1 / scalar), which rounds differently from the kernels'
    __fdiv_rn."""
    xn = (x + BOUND) / torch.full_like(x, 2 * BOUND)
    return xn, xn.clamp(0.0, 1.0), (xn >= 0) & (xn <= 1)


def _cell(x01, scale):
    """locate: pos = x01 * scale + 0.5 (two roundings), lattice cell and fractional weights"""
    pos = x01 * scale + 0.5
    fl = torch.floor(pos)
    return fl.long(), pos - fl


def _corners(lev, base, w):
    """(entry ids [n], fp64 weight [n], fp64 d weight / d w [n, 3]) of the 8 corners, k = x + 2 y + 4 z"""
    from oracle import nerf_oracle as O
    w = w.double()
    fac = (1.0 - w, w)
    for k in range(8):
        b = [(k >> d) & 1 for d in range(3)]
        e = O.hash_corner_index(lev, base[:, 0] + b[0], base[:, 1] + b[1], base[:, 2] + b[2]) + lev.offset
        fx, fy, fz = fac[b[0]][:, 0], fac[b[1]][:, 1], fac[b[2]][:, 2]
        dw = torch.stack([fy * fz * (1 if b[0] else -1), fx * fz * (1 if b[1] else -1), fx * fy * (1 if b[2] else -1)], 1)
        yield e, fx * fy * fz, dw


def _ratio(err, bar):
    """max of err / bar; an error where the bar is zero is infinite"""
    r = torch.where(bar > 0, err / bar.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(r.max()) if r.numel() else 0.0


def _reference(x, tables, lv, gs, anchor_w=None, check_y=None, check_gx=None):
    """fp64 evaluation of the encoder over ``x`` in chunks of CHUNK points.

    tables: flat [E * 2] tables (one, or the three anchors of the tri-blend with per-point weights ``anchor_w`` [P, 3]);
    gs: name -> incoming gradient [P, 2 L].  Returns (G, A): name -> list (per table) of the fp64 table gradient and of
    sum |w g| per element, and the worst ratios of the kernel outputs ``check_y`` (name -> [P, 2 L]) and ``check_gx``
    ((name, g name) -> [P, 3]) against their bars."""
    T = [t.double().view(-1, 2) for t in tables]
    G = {k: [torch.zeros_like(t) for t in T] for k in gs}
    A = {k: [torch.zeros_like(t) for t in T] for k in gs}
    worst = {}
    P = x.shape[0]
    for s in range(0, P, CHUNK):
        e_ = min(P, s + CHUNK)
        n = e_ - s
        _, x01, inside = _x01(x[s:e_])
        aw = anchor_w[s:e_].double() if anchor_w is not None else None
        gc = {k: g[s:e_].double().view(n, len(lv), 2) for k, g in gs.items()}
        y = torch.zeros(n, len(lv), 2, dtype=torch.float64, device=DEV)
        ybar = torch.zeros_like(y)
        gx = {k: torch.zeros(n, 3, dtype=torch.float64, device=DEV) for k in gs}
        gxbar = {k: torch.zeros(n, 3, dtype=torch.float64, device=DEV) for k in gs}
        for l, lev in enumerate(lv):
            base, w = _cell(x01, lev.scale)
            for e, wk, dw in _corners(lev, base, w):
                for i, Ti in enumerate(T):
                    c = wk if aw is None else aw[:, i] * wk
                    te = Ti[e]
                    y[:, l] += c[:, None] * te
                    ybar[:, l] += c[:, None] * te.abs()
                    for k, g in gc.items():
                        contrib = c[:, None] * g[:, l]
                        G[k][i].index_add_(0, e, contrib)
                        A[k][i].index_add_(0, e, contrib.abs())
                        if aw is None:
                            gx[k] += lev.scale * dw * (g[:, l] * te).sum(1, keepdim=True)
                            gxbar[k] += lev.scale * dw.abs() * (g[:, l].abs() * te.abs()).sum(1, keepdim=True)
        y, ybar = y.view(n, -1), ybar.view(n, -1)
        for name, out in (check_y or {}).items():
            worst[name] = max(worst.get(name, 0.0), _ratio((out[s:e_].double() - y).abs(), ybar))
        for (name, k), out in (check_gx or {}).items():
            ref = torch.where(inside, gx[k] / (2 * BOUND), 0.0)
            worst[name, k] = max(worst.get((name, k), 0.0), _ratio((out[s:e_].double() - ref).abs(), gxbar[k] / (2 * BOUND)))
    return G, A, worst


def _table_check(G, G_ref, A, positive):
    """worst |G - G_ref| / A over the elements, and whether the set of touched entries is exact (g > 0 only)"""
    r = _ratio((G.view(-1, 2).double() - G_ref).abs(), A)
    exact = torch.equal(G.view(-1, 2) == 0, A == 0) if positive else True
    return r, exact


# ------------------------------------------------------------------ kernel calls through the C ABI
def _fwd(C, x, P, table, geom, out, ld, col0):
    C.call("b2n_hash_fwd", C.ptr(x), P, BOUND, C.ptr(table), geom.c_levels, L, F, C.ptr(out), ld, col0, C.stream())


def _bwd(C, x, P, table, geom, g, ld, col0, g_table, g_x, lo=0, hi=-1):
    C.call("b2n_hash_bwd", C.ptr(x), P, BOUND, C.ptr(table), geom.c_levels, L, F, C.ptr(g), ld, col0, C.ptr(g_table),
           C.ptr(g_x), 0, lo, hi, C.stream())


def _morton(p):
    """30-bit Morton key of the points (10 bits per axis over the scene box)"""
    def spread(v):
        v = (v | (v << 16)) & 0x030000FF
        v = (v | (v << 8)) & 0x0300F00F
        v = (v | (v << 4)) & 0x030C30C3
        return (v | (v << 2)) & 0x09249249
    q = ((p + BOUND) / (2 * BOUND) * 1023.0).clamp(0, 1023).to(torch.int64)
    return spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2)


class _Env:
    def __init__(self):
        import b2n
        from b2n import march, synthetic
        self.b2n, self.C = b2n, b2n._lib
        ro, rd, _ = synthetic.random_rays(2 ** 18, seed=1)
        u = torch.rand(2 ** 18, 128, generator=torch.Generator().manual_seed(0))
        self.rays = (ro.to(DEV), rd.to(DEV), u.to(DEV))

        def marched(occ):
            return march.march(*self.rays[:2], 2.0, 6.0, 128, self.rays[2], bits=march.pack_occupancy(occ.to(DEV)),
                               R=128, bound=BOUND).pts
        dense = marched(torch.ones(128, 128, 128, dtype=torch.bool))
        ball = marched(synthetic.ball_occupancy(128, BOUND))
        ball = ball[: ball.shape[0] - (ball.shape[0] - 7) % 16].contiguous()       # row count = 7 mod 16
        self.sets = dict(dense=dense, ball=ball, morton=dense[torch.argsort(_morton(dense), stable=True)].contiguous())
        self.refs = {}

    def geometry(self, log2T):
        from oracle import nerf_oracle as O
        geom = self.b2n.HashGeometry(L, 16, 1.5, log2T, F)
        gen = torch.Generator(device=DEV).manual_seed(log2T)
        table = torch.rand(geom.n_params, generator=gen, device=DEV) * 2 - 1
        return geom, O.hash_level_table(L, 16, 1.5, log2T), table

    def grads(self, name):
        P = self.sets[name].shape[0]
        gen = torch.Generator(device=DEV).manual_seed(SEEDS[name])
        pos = 1.0 - torch.rand(P, 2 * L, generator=gen, device=DEV)      # (0, 1]: every contribution nonzero
        sgn = torch.randn(P, 2 * L, generator=gen, device=DEV)
        sgn[::11] = 0.0                                                  # samples that receive no gradient
        return {"pos": pos, "signed": sgn}

    def reference(self, log2T, name, gs=None, **check):
        """(geom, levels, table, G_ref, A) of a geometry and sample set, computed once per module"""
        key = (log2T, name)
        if key not in self.refs or check:
            geom, lv, table = self.geometry(log2T)
            G, A, worst = _reference(self.sets[name], [table], lv, gs or self.grads(name), **check)
            self.refs[key] = (geom, lv, table, {k: v[0] for k, v in G.items()}, {k: v[0] for k, v in A.items()})
            return self.refs[key], worst
        return self.refs[key], {}


@pytest.fixture(scope="module")
def env():
    e = _Env()
    yield e
    e.refs.clear()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------ tests
@pytest.mark.parametrize("log2T", [19, 20])
def test_cell_decisions_match_oracle(env, log2T):
    """The reference's fp32 decisions equal the CPU oracle's fp32 hash_encode arithmetic (which the KAT tests pin to the
    kernels) on a few thousand marched rows and on points placed on cell boundaries, the box faces and outside it: the
    oracle's features rebuilt from these decisions in its own operation order are bit-identical."""
    from oracle import nerf_oracle as O
    geom, lv, table = env.geometry(log2T)
    gen = torch.Generator().manual_seed(5)
    edge = []
    for lev in lv[:6]:                               # lattice planes pos = m + 0.5 ... m + 1, one ulp either side
        m = torch.randint(0, lev.res, (256, 3), generator=gen).float()
        x01 = (m + torch.randint(0, 2, (256, 3), generator=gen).float() * 0.5) / lev.scale
        xw = x01 * (2 * BOUND) - BOUND
        step = torch.randint(-1, 2, (256, 3), generator=gen).float()
        edge.append(torch.nextafter(xw, xw + step * 10))
    faces = torch.tensor([-1.6, -BOUND, -BOUND + 1e-7, 0.0, BOUND - 1e-7, BOUND, 1.6])
    edge.append(faces[torch.randint(0, 7, (512, 3), generator=gen)])
    x = torch.cat([env.sets["dense"][:2048].cpu(), env.sets["ball"][:1024].cpu()] + edge)
    xn, x01, inside = _x01(x.to(DEV))
    xn_cpu = (x + BOUND) / (2 * BOUND)
    assert torch.equal(xn.cpu(), xn_cpu)
    assert torch.equal(inside.cpu(), (xn_cpu >= 0) & (xn_cpu <= 1))
    assert bool((~inside).any()) and bool((x01 == 1).any())
    tab = table.cpu().view(-1, 2)
    y = []
    for lev in lv:                                   # O.hash_encode's loop, fed with the GPU decisions
        base, w = (t.cpu() for t in _cell(x01, lev.scale))
        acc = None
        for k in range(8):
            b = [(k >> d) & 1 for d in range(3)]
            wt = None
            for d in range(3):
                wd = w[:, d] if b[d] else (1.0 - w[:, d])
                wt = wd if wt is None else wt * wd
            term = wt[:, None] * tab[O.hash_corner_index(lev, base[:, 0] + b[0], base[:, 1] + b[1], base[:, 2] + b[2])
                                     + lev.offset]
            acc = term if acc is None else acc + term
        y.append(acc)
    assert torch.equal(torch.cat(y, -1), O.hash_representation(x, table.cpu(), lv, F, BOUND))


@pytest.mark.parametrize("sample_set", ["dense", "ball", "morton"])
@pytest.mark.parametrize("log2T", [19, 20])
def test_hash_grid_vs_fp64_every_config(env, log2T, sample_set):
    """Features, input gradient and table gradient of every kernel configuration at training size.  T = 2^19 is the C2
    geometry (level 4 hashed, the forward's staged store on); at T = 2^20 level 4 is dense and the 94 MB table turns the
    staged store off."""
    C = env.C
    x = env.sets[sample_set]
    P = x.shape[0]
    geom, lv, table = env.geometry(log2T)
    gs = env.grads(sample_set)
    ys, gxs = {}, {}
    for fwd in (0, 1):                               # variant bit 0: forward and input-gradient kernels
        with C.hash_variant(fwd | 2, 128):
            ys[f"fwd{fwd}"] = torch.empty(P, 2 * L, device=DEV)
            _fwd(C, x, P, table, geom, ys[f"fwd{fwd}"], 2 * L, 0)
            for k, g in gs.items():
                gxs[f"fwd{fwd}", k] = torch.empty(P, 3, device=DEV)
                _bwd(C, x, P, table, geom, g, 2 * L, 0, None, gxs[f"fwd{fwd}", k])
    (geom, lv, table, G_ref, A), worst = env.reference(log2T, sample_set, gs, check_y=ys, check_gx=gxs)
    del ys, gxs
    bad = []
    for fwd in (0, 1):
        r = record(f"hash_fullsize[T{log2T}]:features/bar[fwd{fwd}]", worst[f"fwd{fwd}"])
        if not r <= TOL_Y:
            bad.append(("features", fwd, r))
        for k in gs:
            r = record(f"hash_fullsize[T{log2T}]:g_x/bar[fwd{fwd}]", worst[f"fwd{fwd}", k])
            if not r <= TOL_X:
                bad.append(("g_x", fwd, k, r))
    G = torch.empty(geom.n_params, device=DEV)
    for variant, merge in CONFIGS:
        with C.hash_variant(variant, merge):
            for k, g in gs.items():
                G.zero_()
                _bwd(C, x, P, table, geom, g, 2 * L, 0, G, None)
                r, exact = _table_check(G, G_ref[k], A[k], k == "pos")
                record(f"hash_fullsize[T{log2T}]:g_table/A[v{variant},m{merge}]", r)
                if not (r <= TOL_G and exact):
                    bad.append(("g_table", variant, merge, k, r, exact))
    assert not bad, bad


@pytest.mark.parametrize("split", [4, 8])
@pytest.mark.parametrize("log2T", [19, 20])
def test_level_windows_add_up(env, log2T, split):
    """The data-parallel split (b2n.ops: the fine levels are scattered first, then the coarse ones with g_x): each window
    writes its own levels only, and the two together meet the per-element bar; g_x does not depend on the window."""
    C = env.C
    x = env.sets["dense"]
    P = x.shape[0]
    (geom, lv, table, G_ref, A), _ = env.reference(log2T, "dense")
    g = env.grads("dense")["signed"]
    cut = lv[split].offset * F
    gx_full = torch.empty(P, 3, device=DEV)
    _bwd(C, x, P, table, geom, g, 2 * L, 0, None, gx_full)
    G = torch.zeros(geom.n_params, device=DEV)
    gx = torch.empty(P, 3, device=DEV)
    _bwd(C, x, P, table, geom, g, 2 * L, 0, G, None, split, L)
    assert float(G[:cut].abs().max()) == 0.0 and float(G[cut:].abs().max()) > 0.0
    _bwd(C, x, P, table, geom, g, 2 * L, 0, G, gx, 0, split)
    r, _ = _table_check(G, G_ref["signed"], A["signed"], False)
    assert record(f"hash_fullsize[T{log2T}]:g_table/A[window {split}]", r) <= TOL_G
    assert torch.equal(gx, gx_full)


@pytest.mark.parametrize("variant", [0, 1, 2, 3])
@pytest.mark.parametrize("log2T", [19, 20])
def test_static_capacity_rows_behind_the_count(env, log2T, variant):
    """include/b2nerf.h b2n_set_active_rows: with the ball set in a capacity buffer (2^25 rows, device-side count = 7 mod 16)
    and finite garbage positions / NaN gradients behind the count, the table gradient is that of the counted rows, the
    counted rows of out / g_x equal the unbounded call's, and every row behind the count keeps its sentinel."""
    C = env.C
    (geom, lv, table, G_ref, A), _ = env.reference(log2T, "ball")
    x = env.sets["ball"]
    n = x.shape[0]
    cap = 2 ** 18 * 128
    assert n % 16 and n < cap
    gen = torch.Generator(device=DEV).manual_seed(7)
    xc = torch.rand(cap, 3, generator=gen, device=DEV) * 4 - 2
    xc[:n] = x
    sentinel = -12345.0
    g = env.grads("ball")["pos"]
    gc = torch.full((cap, 2 * L), math.nan, device=DEV)
    gc[:n] = g
    n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
    with C.hash_variant(variant, SHIPPED[1]):
        y0, gx0 = torch.empty(n, 2 * L, device=DEV), torch.empty(n, 3, device=DEV)
        _fwd(C, x, n, table, geom, y0, 2 * L, 0)
        _bwd(C, x, n, table, geom, g, 2 * L, 0, None, gx0)
        out = torch.full((cap, 2 * L), sentinel, device=DEV)
        gx = torch.full((cap, 3), sentinel, device=DEV)
        G = torch.zeros(geom.n_params, device=DEV)
        with C.active_rows(n_dev):
            _fwd(C, xc, cap, table, geom, out, 2 * L, 0)
            _bwd(C, xc, cap, table, geom, gc, 2 * L, 0, G, gx)
    assert torch.equal(out[:n], y0) and bool((out[n:] == sentinel).all())
    assert torch.equal(gx[:n], gx0) and bool((gx[n:] == sentinel).all())
    r, exact = _table_check(G, G_ref["pos"], A["pos"], True)
    assert record(f"hash_fullsize[T{log2T}]:g_table/A[static capacity]", r) <= TOL_G and exact


@pytest.mark.parametrize("variant", [0, 1, 2, 3])
def test_strided_rows(env, variant):
    """out and g as columns 3 .. 34 of 37-wide rows (the non-vector load / store paths): the same features and g_x as the
    contiguous call, the columns around them untouched / never read (NaN there), and the table gradient within the bar."""
    C = env.C
    (geom, lv, table, G_ref, A), _ = env.reference(19, "ball")
    x = env.sets["ball"]
    n = x.shape[0]
    ld, col0 = 37, 3
    g = env.grads("ball")["signed"]
    gw = torch.full((n, ld), math.nan, device=DEV)
    gw[:, col0:col0 + 2 * L] = g
    with C.hash_variant(variant, SHIPPED[1]):
        y0, gx0 = torch.empty(n, 2 * L, device=DEV), torch.empty(n, 3, device=DEV)
        _fwd(C, x, n, table, geom, y0, 2 * L, 0)
        _bwd(C, x, n, table, geom, g, 2 * L, 0, None, gx0)
        out = torch.full((n, ld), -7.0, device=DEV)
        gx = torch.empty(n, 3, device=DEV)
        G = torch.zeros(geom.n_params, device=DEV)
        _fwd(C, x, n, table, geom, out, ld, col0)
        _bwd(C, x, n, table, geom, gw, ld, col0, G, gx)
    assert torch.equal(out[:, col0:col0 + 2 * L], y0)
    assert bool((out[:, :col0] == -7.0).all()) and bool((out[:, col0 + 2 * L:] == -7.0).all())
    assert torch.equal(gx, gx0)
    r, _ = _table_check(G, G_ref["signed"], A["signed"], False)
    assert record("hash_fullsize[T19]:g_table/A[strided]", r) <= TOL_G


def test_tri_blend_vs_fp64(env):
    """b2n_hash_tri_fwd / _bwd at the C5 deformation geometry (L = 12, T = 2^16) on about 8 M marched points with per-ray
    times (t = 0, 0.5, 1 included, where anchors drop out).  The tent weights are formed in fp32 in tri_weights' order."""
    from b2n import march
    from oracle import nerf_oracle as O
    b2n, C = env.b2n, env.C
    B = 88000
    ro, rd, u = (t[:B] for t in env.rays)
    tr = torch.rand(B, 1, generator=torch.Generator().manual_seed(8))
    tr[0::7], tr[1::7], tr[2::7] = 0.0, 0.5, 1.0
    m = march.march(ro, rd, 2.0, 6.0, 128, u, bits=march.pack_occupancy(torch.ones(128, 128, 128, dtype=torch.bool,
                    device=DEV)), R=128, bound=BOUND, times=tr.to(DEV))
    x, t = m.pts, m.times.reshape(-1)
    P = x.shape[0]
    Lt = 12
    geom = b2n.HashGeometry(Lt, 16, 1.5, 16, 2)
    lv = O.hash_level_table(Lt, 16, 1.5, 16)
    gen = torch.Generator(device=DEV).manual_seed(16)
    tabs = [torch.rand(geom.n_params, generator=gen, device=DEV) * 2 - 1 for _ in range(3)]
    w = [torch.clamp(1.0 - torch.abs(t - a) / 0.5, 0.0, 1.0) for a in (0.0, 0.5, 1.0)]
    tot = w[0] + w[1] + w[2] + 1e-8
    aw = torch.stack([wi / tot for wi in w], 1)
    pos = 1.0 - torch.rand(P, 2 * Lt, generator=gen, device=DEV)
    sgn = torch.randn(P, 2 * Lt, generator=gen, device=DEV)
    sgn[::11] = 0.0
    gs = {"pos": pos, "signed": sgn}
    y = torch.empty(P, 2 * Lt, device=DEV)
    C.call("b2n_hash_tri_fwd", C.ptr(x), C.ptr(t), P, BOUND, *(C.ptr(tb) for tb in tabs), geom.c_levels, Lt, C.ptr(y),
           2 * Lt, C.stream())
    G_ref, A, worst = _reference(x, tabs, lv, gs, anchor_w=aw, check_y={"tri": y})
    bad = []
    if not record("hash_fullsize[tri]:features/bar", worst["tri"]) <= TOL_Y:
        bad.append(("features", worst["tri"]))
    for k, g in gs.items():
        grads = [torch.zeros(geom.n_params, device=DEV) for _ in range(3)]
        C.call("b2n_hash_tri_bwd", C.ptr(x), C.ptr(t), P, BOUND, geom.c_levels, Lt, C.ptr(g), 2 * Lt,
               *(C.ptr(gr) for gr in grads), C.stream())
        for i in range(3):
            r, exact = _table_check(grads[i], G_ref[k][i], A[k][i], k == "pos")
            record("hash_fullsize[tri]:g_table/A", r)
            if not (r <= TOL_G and exact):
                bad.append(("g_table", i, k, r, exact))
    assert not bad, bad


def test_shipped_configuration_restored(env):
    """every switch above restored what it found: later tests run the shipped kernels"""
    assert env.C.hash_config() == SHIPPED
