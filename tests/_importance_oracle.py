"""float64 restatement of the hierarchical-sampling contract (b2n_importance_sample of include/b2nerf.h, DESIGN.md §5h):
NeRF's sample_pdf over the coarse compositing weights, then the stable merge of the coarse and fine depths."""
import numpy as np


def weights(sigma, z, dnorm):
    """compositing weights [B,Nc]: delta = (z_{s+1} - z_s)|d| (1e10 |d| last), alpha = 1 - exp(-sigma delta),
    w = alpha * prod_{j<s} (1 - alpha_j + 1e-10)"""
    sigma, z = np.asarray(sigma, np.float64), np.asarray(z, np.float64)
    delta = np.concatenate([z[:, 1:] - z[:, :-1], np.full((z.shape[0], 1), 1e10)], -1) * np.asarray(dnorm)[:, None]
    alpha = -np.expm1(-sigma * delta)
    trans = np.cumprod(np.concatenate([np.ones((z.shape[0], 1)), 1.0 - alpha[:, :-1] + 1e-10], -1), -1)
    return alpha * trans


def cdf_of(w):
    """[B,Nc-1]: c = [0, cumsum(pdf)] of the interior weights w_1 .. w_{Nc-2}, each + 1e-5; the last entry is exactly 1
    (so that u = 1 is past every breakpoint, not on one side or the other of a rounded sum)"""
    wi = w[:, 1:-1] + 1e-5
    pdf = wi / wi.sum(-1, keepdims=True)
    cdf = np.concatenate([np.zeros((w.shape[0], 1)), np.cumsum(pdf, -1)], -1)
    cdf[:, -1] = 1.0
    return cdf


def u_stratified(U):
    """u_k = (k + U_k) / Nf"""
    U = np.asarray(U, np.float64)
    return (np.arange(U.shape[1]) + U) / U.shape[1]


def invert(cdf, mids, u, flat=1e-5):
    """inverse CDF of the contract; returns (z_fine [B,Nf], denom [B,Nf] before the flat-bin replacement,
    m[above] - m[below] [B,Nf])"""
    B, nb = cdf.shape
    z_fine = np.empty(u.shape)
    denom = np.empty(u.shape)
    width = np.empty(u.shape)
    for r in range(B):
        i = np.searchsorted(cdf[r], u[r], side="right")
        below = np.maximum(i - 1, 0)
        above = np.minimum(i, nb - 1)
        d = cdf[r, above] - cdf[r, below]
        denom[r] = d
        width[r] = mids[r, above] - mids[r, below]
        d = np.where(d < flat, 1.0, d)
        t = (u[r] - cdf[r, below]) / d
        z_fine[r] = mids[r, below] + t * (mids[r, above] - mids[r, below])
    return z_fine, denom, width


def bracket(cdf, mids, u, eps, flat=1e-5, flat_rel=0.0):
    """(lo, hi) [B,Nf]: the range of the inverse CDF over positions within eps of u and flat-bin thresholds within
    flat_rel of ``flat`` -- every value a CDF rounded by up to eps can give.  The inverse CDF is non-decreasing in u, so
    the extremes are at the ends of the range."""
    outs = [invert(cdf, mids, u + du, flat * (1 + df))[0] for du in (-eps, 0.0, eps) for df in (-flat_rel, flat_rel)]
    return np.min(outs, 0), np.max(outs, 0)


def sample(sigma, z, dnorm, u, flat=1e-5):
    """fine depths [B,Nf] for the positions u [B,Nf] (non-decreasing per ray); also returns the CDF and the midpoints"""
    z = np.asarray(z, np.float64)
    mids = 0.5 * (z[:, 1:] + z[:, :-1])
    cdf = cdf_of(weights(sigma, z, dnorm))
    z_fine = invert(cdf, mids, np.asarray(u, np.float64), flat)[0]
    return z_fine, cdf, mids


def merge(z, z_fine):
    """(z_merged [B,Nc+Nf], merge_src [B,Nc+Nf]): the stable merge of the sorted coarse and fine depths, coarse first on
    ties; source s for coarse slot s, Nc + k for fine slot k"""
    both = np.concatenate([z, z_fine], -1)
    src = np.argsort(both, axis=-1, kind="stable")
    return np.take_along_axis(both, src, -1), src.astype(np.int32)
