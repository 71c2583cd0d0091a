"""float64 / integer restatement of the error-map contract (b2n_errormap_* of include/b2nerf.h, DESIGN.md §5i): the
update, the CDF in the kernel's fixed association, the inverse mapping u -> pixel, and the ratio 1 / (N p)."""
import numpy as np

RUN, THREADS = 16, 256                  # cells per run, runs per block of the CDF's association


def cell_bounds(H, Hm):
    """first pixel row of every cell row and one past its last: [ceil(i H / Hm), ceil((i+1) H / Hm))"""
    i = np.arange(Hm + 1, dtype=np.int64)
    b = (i * H + Hm - 1) // Hm
    return b[:-1], b[1:]


def cell_of(v, y, x, H, W, Hm, Wm):
    return (v * Hm + y * Hm // H) * Wm + x * Wm // W


def update(e, picks, err, beta, H, W):
    """the map after one update: integer sums of rint(clip(err) 2^24) and counts per cell, then the fp32 momentum"""
    e = np.asarray(e, np.float32)
    V, Hm, Wm = e.shape
    v, y, x = (np.clip(np.asarray(p, np.int64), 0, hi - 1) for p, hi in zip(picks, (V, H, W)))
    err = np.asarray(err, np.float32)
    s = np.where(np.isfinite(err), np.clip(err, np.float32(0), np.float32(1)), np.float32(0)).astype(np.float32)
    q = np.rint(s.astype(np.float64) * 2.0 ** 24).astype(np.uint64)
    c = cell_of(v, y, x, H, W, Hm, Wm)
    n = V * Hm * Wm
    sums = np.zeros(n, np.uint64)
    np.add.at(sums, c, q)
    cnt = np.bincount(c, minlength=n).astype(np.int64)
    flat = e.ravel().copy()
    hit = cnt > 0
    m = (sums[hit].astype(np.float64) * 2.0 ** -24 / cnt[hit]).astype(np.float32)
    old = flat[hit]
    b = np.float32(beta)
    flat[hit] = np.where(old < 0, m, (np.float32(1) - b) * old + b * m)
    return flat.reshape(e.shape)


def weights(e):
    e = np.asarray(e, np.float32).ravel()
    return np.where(e > 0, e, np.float32(0)).astype(np.float64)            # NaN -> 0


def cdf(e):
    """the inclusive fp64 prefix of the weights in the kernel's association: running sums over runs of 16 cells, the
    runs of a 4096-cell block chained in order, the blocks chained in order (np.cumsum adds sequentially)"""
    w = weights(e)
    n = w.size
    nb = -(-n // (RUN * THREADS))
    wp = np.zeros(nb * RUN * THREADS)
    wp[:n] = w
    run = np.cumsum(wp.reshape(nb, THREADS, RUN), axis=-1)
    tot = run[..., -1]
    excl = np.zeros_like(tot)
    excl[:, 1:] = np.cumsum(tot, axis=-1)[:, :-1]
    block = excl[:, -1] + tot[:, -1]
    off = np.zeros(nb)
    off[1:] = np.cumsum(block)[:-1]
    return (off[:, None, None] + (excl[:, :, None] + run)).ravel()[:n]


def _floor_index(f, n):
    with np.errstate(invalid="ignore"):
        x = np.floor(f * np.float64(n))
        ok = x >= 0
    x = np.where(ok, x, 0.0)
    return np.where(x >= n - 1, n - 1, x).astype(np.int64)


def sample(e, c, u, lam, H, W):
    """(img_idx, pix_y, pix_x, ratio) for the uniforms u [B,3] (fp32) and the CDF c of the map e"""
    V, Hm, Wm = np.asarray(e).shape
    n, N = V * Hm * Wm, V * H * W
    lam32 = np.float32(lam)
    L = np.float64(lam32)
    S = c[-1]
    use_map = bool(lam32 < 1 and 0 < S < np.inf)
    u = np.asarray(u, np.float32).astype(np.float64)
    u0, u1, u2 = u[:, 0], u[:, 1], u[:, 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        uni = (u0 < L) | (not use_map)
        k = _floor_index(u0 / L if use_map else u0, N)
        t = (u0 - L) / (1.0 - L) * S if use_map else np.zeros_like(u0)
        fwd = t < S
    cell = np.where(fwd, np.minimum(np.searchsorted(c, np.where(fwd, t, 0.0), side="right"), n - 1),
                    min(int(np.searchsorted(c, S, side="left")), n - 1))
    cv, ci, cj = cell // (Hm * Wm), (cell // Wm) % Hm, cell % Wm
    ylo, yhi = cell_bounds(H, Hm)
    xlo, xhi = cell_bounds(W, Wm)
    my = ylo[ci] + _floor_index(u1, yhi[ci] - ylo[ci])
    mx = xlo[cj] + _floor_index(u2, xhi[cj] - xlo[cj])
    v = np.where(uni, k // (H * W), cv)
    y = np.where(uni, (k % (H * W)) // W, my)
    x = np.where(uni, k % W, mx)
    return v, y, x, ratio(e, lam, H, W, v, y, x)


def prob(e, lam, H, W):
    """the sampling probability of every pixel [V,H,W], stated directly: lam / N + (1 - lam) w_c / (S |cell c|) with the
    cell sizes counted, not derived from the ceil formula; uniform when the map carries no finite positive mass"""
    e = np.asarray(e, np.float32)
    V, Hm, Wm = e.shape
    N = V * H * W
    L = np.float64(np.float32(lam))
    w = weights(e)
    S = w.sum()
    if not (L < 1 and 0 < S < np.inf):
        return np.full((V, H, W), 1.0 / N)
    v, y, x = np.meshgrid(np.arange(V), np.arange(H), np.arange(W), indexing="ij")
    c = cell_of(v, y, x, H, W, Hm, Wm)
    size = np.bincount(c.ravel(), minlength=w.size)
    return L / N + (1 - L) * w[c] / (S * size[c])


def ratio(e, lam, H, W, v, y, x):
    """1 / (N p) of the picks, fp32"""
    V = np.asarray(e).shape[0]
    return (1.0 / (V * H * W * prob(e, lam, H, W)[v, y, x])).astype(np.float32)
