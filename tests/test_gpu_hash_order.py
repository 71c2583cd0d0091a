"""The spatially ordered hash-grid path (include/b2nerf.h b2n_hash_order, b2n_hash_fwd_ordered / b2n_hash_bwd_ordered) at
C2 training size, on the dense and ball sample sets of test_gpu_hash_fullsize and against its fp64 reference:

* the order is a permutation whose Morton keys (2^7 lattice) do not decrease, and x_sorted = x[order];
* features through the order are bitwise those of the plain entry: contiguous, strided rows, and static capacity (a
  device-side count off every multiple of 16, garbage rows behind it whose sentinels survive);
* the table gradient is within 1e-4 of sum |w g| per element with the shipped merging and with merging off, touches
  exactly the entries a positive gradient reaches, and the level windows [0,4)+[4,16) add up;
* hash_encode orders large inputs itself, also inside a captured CUDA graph with a device-side row count."""
import math

import pytest
import torch

from _util import record
from test_gpu_hash_fullsize import BOUND, DEV, F, L, SHIPPED, TOL_G, _Env, _table_check

pytestmark = pytest.mark.gpu
BITS = 7


@pytest.fixture(scope="module")
def env():
    e = _Env()
    yield e
    e.refs.clear()
    torch.cuda.empty_cache()


def _key(x):
    """the kernels' bucket: Morton code of the cell of clamp((x + b) / 2b, 0, 1) on a 2^BITS lattice"""
    u = ((x + BOUND) / torch.full_like(x, 2 * BOUND)).clamp(0.0, 1.0)
    q = (u * (1 << BITS)).to(torch.int64).clamp_max((1 << BITS) - 1)
    key = torch.zeros(x.shape[0], dtype=torch.int64, device=x.device)
    for b in range(BITS):
        for d in range(3):
            key |= ((q[:, d] >> b) & 1) << (3 * b + d)
    return key


def _order(C, x, P):
    order = torch.full((P,), -1, dtype=torch.int32, device=DEV)
    xs = torch.empty_like(x)
    scratch = torch.empty(C.lib.b2n_hash_order_scratch(P) // 4, dtype=torch.int32, device=DEV)
    C.call("b2n_hash_order", C.ptr(x), P, BOUND, C.ptr(order), C.ptr(xs), C.ptr(scratch), C.stream())
    return order, xs


def _fwd(C, x, order, P, table, geom, out, ld, col0):
    if order is None:
        C.call("b2n_hash_fwd", C.ptr(x), P, BOUND, C.ptr(table), geom.c_levels, L, F, C.ptr(out), ld, col0, C.stream())
    else:
        C.call("b2n_hash_fwd_ordered", C.ptr(x), C.ptr(order), P, BOUND, C.ptr(table), geom.c_levels, L, F, C.ptr(out),
               ld, col0, C.stream())


def _bwd_ordered(C, xs, order, P, table, geom, g, ld, col0, G, lo=0, hi=-1):
    C.call("b2n_hash_bwd_ordered", C.ptr(xs), C.ptr(order), P, BOUND, C.ptr(table), geom.c_levels, L, F, C.ptr(g), ld,
           col0, C.ptr(G), lo, hi, C.stream())


@pytest.mark.parametrize("sample_set", ["dense", "ball"])
def test_order_is_a_sorted_permutation(env, sample_set):
    x = env.sets[sample_set]
    P = x.shape[0]
    order, xs = _order(env.C, x, P)
    o = order.long()
    assert torch.equal(torch.sort(o).values, torch.arange(P, device=DEV))
    assert bool((_key(x)[o].diff() >= 0).all())
    assert torch.equal(xs, x[o])


@pytest.mark.parametrize("sample_set", ["dense", "ball"])
def test_ordered_features_and_table_gradient(env, sample_set):
    C = env.C
    x = env.sets[sample_set]
    P = x.shape[0]
    (geom, lv, table, G_ref, A), _ = env.reference(19, sample_set)
    order, xs = _order(C, x, P)
    y0, y1 = torch.empty(P, 2 * L, device=DEV), torch.empty(P, 2 * L, device=DEV)
    _fwd(C, x, None, P, table, geom, y0, 2 * L, 0)
    _fwd(C, xs, order, P, table, geom, y1, 2 * L, 0)
    assert torch.equal(y0, y1)
    G = torch.empty(geom.n_params, device=DEV)
    bad = []
    for merge in (SHIPPED[1], 0):
        with C.hash_variant(SHIPPED[0], merge):
            for k, g in env.grads(sample_set).items():
                G.zero_()
                _bwd_ordered(C, xs, order, P, table, geom, g, 2 * L, 0, G)
                r, exact = _table_check(G, G_ref[k], A[k], k == "pos")
                record(f"hash_order[{sample_set}]:g_table/A[m{merge},{k}]", r)
                if not (r <= TOL_G and exact):
                    bad.append((merge, k, r, exact))
    assert not bad, bad


def test_ordered_level_windows_add_up(env):
    C = env.C
    x = env.sets["dense"]
    P = x.shape[0]
    (geom, lv, table, G_ref, A), _ = env.reference(19, "dense")
    g = env.grads("dense")["signed"]
    order, xs = _order(C, x, P)
    cut = lv[4].offset * F
    G = torch.zeros(geom.n_params, device=DEV)
    _bwd_ordered(C, xs, order, P, table, geom, g, 2 * L, 0, G, 4, L)
    assert float(G[:cut].abs().max()) == 0.0 and float(G[cut:].abs().max()) > 0.0
    _bwd_ordered(C, xs, order, P, table, geom, g, 2 * L, 0, G, 0, 4)
    r, _ = _table_check(G, G_ref["signed"], A["signed"], False)
    assert record("hash_order[dense]:g_table/A[window 4]", r) <= TOL_G


def test_ordered_static_capacity_and_strided_rows(env):
    """ball set in a 2^25-row capacity buffer (device-side count = 7 mod 16, garbage positions and NaN gradients behind
    it), then as columns 3 .. 34 of 37-wide rows"""
    C = env.C
    (geom, lv, table, G_ref, A), _ = env.reference(19, "ball")
    x = env.sets["ball"]
    n = x.shape[0]
    cap = 2 ** 18 * 128
    assert n % 16 and n < cap
    y0 = torch.empty(n, 2 * L, device=DEV)
    _fwd(C, x, None, n, table, geom, y0, 2 * L, 0)
    gen = torch.Generator(device=DEV).manual_seed(7)
    xc = torch.rand(cap, 3, generator=gen, device=DEV) * 4 - 2
    xc[:n] = x
    g = env.grads("ball")["pos"]
    gc = torch.full((cap, 2 * L), math.nan, device=DEV)
    gc[:n] = g
    sentinel = -12345.0
    n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
    out = torch.full((cap, 2 * L), sentinel, device=DEV)
    G = torch.zeros(geom.n_params, device=DEV)
    with C.active_rows(n_dev):
        order, xs = _order(C, xc, cap)
        _fwd(C, xs, order, cap, table, geom, out, 2 * L, 0)
        _bwd_ordered(C, xs, order, cap, table, geom, gc, 2 * L, 0, G)
    assert torch.equal(order[n:].long(), torch.arange(n, cap, device=DEV))        # rows behind the count stay put
    assert torch.equal(torch.sort(order[:n].long()).values, torch.arange(n, device=DEV))
    assert torch.equal(out[:n], y0) and bool((out[n:] == sentinel).all())
    r, exact = _table_check(G, G_ref["pos"], A["pos"], True)
    assert record("hash_order[ball]:g_table/A[static capacity]", r) <= TOL_G and exact

    ld, col0 = 37, 3
    order, xs = _order(C, x, n)
    gs = env.grads("ball")["signed"]
    gw = torch.full((n, ld), math.nan, device=DEV)
    gw[:, col0:col0 + 2 * L] = gs
    out = torch.full((n, ld), -7.0, device=DEV)
    G.zero_()
    _fwd(C, xs, order, n, table, geom, out, ld, col0)
    _bwd_ordered(C, xs, order, n, table, geom, gw, ld, col0, G)
    assert torch.equal(out[:, col0:col0 + 2 * L], y0)
    assert bool((out[:, :col0] == -7.0).all()) and bool((out[:, col0 + 2 * L:] == -7.0).all())
    r, _ = _table_check(G, G_ref["signed"], A["signed"], False)
    assert record("hash_order[ball]:g_table/A[strided]", r) <= TOL_G


def test_ordered_entries_refuse_what_they_cannot_run(env):
    C = env.C
    x = env.sets["ball"][:4096]
    geom, lv, table = env.geometry(19)
    order, xs = _order(C, x, 4096)
    out = torch.empty(4096, 2 * L, device=DEV)
    with C.hash_variant(0, SHIPPED[1]):
        with pytest.raises(ValueError, match="b2n_hash_fwd_ordered"):
            _fwd(C, xs, order, 4096, table, geom, out, 2 * L, 0)
        with pytest.raises(ValueError, match="b2n_hash_bwd_ordered"):
            _bwd_ordered(C, xs, order, 4096, table, geom, out, 2 * L, 0, torch.zeros_like(table))


def test_hash_encode_orders_inside_a_cuda_graph(env):
    """hash_encode above HASH_ORDER_MIN_POINTS goes through the ordered entries; one forward + backward captured as a CUDA
    graph over a capacity buffer with a device-side row count gives the eager plain path's features and a table gradient
    within the per-element bar."""
    import b2n
    from b2n import ops
    C = env.C
    x = env.sets["dense"]
    n = x.shape[0]
    assert n >= ops.HASH_ORDER_MIN_POINTS
    (geom, lv, table0, G_ref, A), _ = env.reference(19, "dense")
    g = env.grads("dense")["pos"]
    y0 = torch.empty(n, 2 * L, device=DEV)
    _fwd(C, x, None, n, table0, geom, y0, 2 * L, 0)
    cap = n + 1000
    xc = torch.zeros(cap, 3, device=DEV)
    xc[:n] = x
    gc = torch.zeros(cap, 2 * L, device=DEV)
    gc[:n] = g
    n_dev = torch.tensor([n], dtype=torch.int32, device=DEV)
    table = table0.clone().requires_grad_(True)
    calls = []
    real_call = C.call
    C.call = lambda name, *a, **k: (calls.append(name), real_call(name, *a, **k))[1]
    def step():
        # the forward under the device-side count, the backward outside it: the backward runs on autograd's thread and
        # re-installs the forward's count there itself (b2n._lib.with_ctx_rows)
        table.grad = None
        with C.active_rows(n_dev):
            y = b2n.hash_encode(xc, table, geom, BOUND)
        y.backward(gc)
        return y

    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            step()                                                # warm-up outside the capture
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            y = step()
        graph.replay()
        torch.cuda.synchronize()
    finally:
        C.call = real_call
    assert "b2n_hash_order" in calls and "b2n_hash_fwd_ordered" in calls and "b2n_hash_bwd_ordered" in calls
    assert torch.equal(y[:n], y0)
    r, exact = _table_check(table.grad, G_ref["pos"], A["pos"], True)
    assert record("hash_order[dense]:g_table/A[cuda graph]", r) <= TOL_G and exact
