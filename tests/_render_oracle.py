"""float64 numpy restatement of the fast-render contract (b2n.render, include/b2nerf.h b2n_render_*, DESIGN.md §5g):
the active samples of every ray composited front to back, one at a time, and a ray stops after the first sample that
leaves its transmittance T below eps."""
import numpy as np


def render(sigma, rgb, z, dnorm, active, eps, bg):
    """sigma [B,N], rgb [B,N,3], z [N] (the depths, shared by every ray), dnorm [B] (|d|), active [B,N] bool,
    eps >= 0, bg [3] or [B,3].  Returns (color [B,3], depth [B], acc [B], n [B] composited samples per ray,
    gap = min over composited samples of |T / eps - 1| after the sample (inf for eps = 0)).

    delta_s = (z[s+1] - z[s]) * |d|, 1e10 * |d| for the last sample; alpha = 1 - exp(-sigma * delta); w = alpha * T;
    T <- T * (1 - alpha + 1e-10).  N == 1 composites nothing (the reference's empty interval tensor)."""
    sigma, rgb, z = np.asarray(sigma, np.float64), np.asarray(rgb, np.float64), np.asarray(z, np.float64)
    dnorm, active = np.asarray(dnorm, np.float64), np.asarray(active, bool)
    B, N = sigma.shape
    T = np.ones(B)
    color, depth, acc = np.zeros((B, 3)), np.zeros(B), np.zeros(B)
    n = np.zeros(B, np.int64)
    alive = np.ones(B, bool)
    gap = np.inf
    for s in range(N if N > 1 else 0):
        delta = ((z[s + 1] - z[s]) if s < N - 1 else 1e10) * dnorm
        alpha = 1.0 - np.exp(-sigma[:, s] * delta)
        m = alive & active[:, s]
        w = np.where(m, alpha * T, 0.0)
        color += w[:, None] * rgb[:, s]
        depth += w * z[s]
        acc += w
        T = np.where(m, T * (1.0 - alpha + 1e-10), T)
        n += m
        if eps > 0 and m.any():
            gap = min(gap, float(np.abs(T[m] / eps - 1.0).min()))
            alive &= ~(m & (T < eps))
    bg = np.asarray(bg, np.float64)
    color = color + (1.0 - acc)[:, None] * (bg[None] if bg.ndim == 1 else bg)
    return color, depth, acc, n, gap
