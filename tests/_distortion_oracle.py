"""float64 restatement of the distortion-loss contract (b2n_distortion_* of include/b2nerf.h, DESIGN.md §5j): the
mip-NeRF 360 double sum (Barron et al. 2022, eq. 15) over the compositing weights, its gradient w.r.t. sigma by
autograd, and the O(N) prefix-sum form with its closed-form dL/dw that the kernels use.  Device-agnostic torch."""
import torch


def weights(sigma, z, dnorm):
    """compositing weights [B,N]: tau = (z_{i+1} - z_i)|d| (1e10 |d| last), alpha = 1 - exp(-sigma tau),
    w = alpha * prod_{j<i} (1 - alpha_j + 1e-10)"""
    tau = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1) * dnorm[:, None]
    alpha = 1.0 - torch.exp(-sigma * tau)
    trans = torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1.0 - alpha[:, :-1] + 1e-10], -1), -1)
    return alpha * trans


def intervals(z, near, far):
    """(midpoint, width) [B,N] of [s_i, s_{i+1}] in s = (z - near) / (far - near), s_N = 1"""
    s = (z - near) / (far - near)
    s_next = torch.cat([s[:, 1:], torch.ones_like(s[:, :1])], -1)
    return 0.5 * (s + s_next), s_next - s


def loss_of_weights(w, mid, width):
    """the double sum: sum_ij w_i w_j |m_i - m_j| + 1/3 sum_i w_i^2 d_i  [B]"""
    pair = (w[:, :, None] * w[:, None, :] * (mid[:, :, None] - mid[:, None, :]).abs()).sum((1, 2))
    return pair + (w * w * width).sum(-1) / 3.0


def loss(sigma, z, rays_d, near, far):
    """loss [B] (float64) of dense sigma [B,N] (inactive samples: sigma = 0)"""
    sigma, z, rays_d = sigma.double(), z.double(), rays_d.double()
    w = weights(sigma, z, rays_d.norm(dim=-1))
    mid, width = intervals(z, float(near), float(far))
    return loss_of_weights(w, mid, width)


def loss_and_grad(sigma, z, rays_d, near, far, g_loss=None):
    """(loss [B], dL/dsigma [B,N] of sum_r g_loss[r] * loss[r]) in float64, the gradient by autograd"""
    s = sigma.detach().double().requires_grad_(True)
    L = loss(s, z, rays_d, near, far)
    g = torch.ones_like(L) if g_loss is None else g_loss.double()
    gs, = torch.autograd.grad((L * g).sum(), s)
    return L.detach(), gs


def prefix_form(w, mid, width):
    """the O(N) form of the kernels: 2 sum_i w_i (m_i W_{<i} - WM_{<i}) + 1/3 sum_i w_i^2 d_i"""
    wm = w * mid
    W_ex = torch.cumsum(w, -1) - w
    WM_ex = torch.cumsum(wm, -1) - wm
    return 2.0 * (w * (mid * W_ex - WM_ex)).sum(-1) + (w * w * width).sum(-1) / 3.0


def grad_w(w, mid, width):
    """dL/dw_i = 2 (m_i W_{<i} - WM_{<i} + WM_{>i} - m_i W_{>i}) + 2/3 w_i d_i"""
    wm = w * mid
    W_in, WM_in = torch.cumsum(w, -1), torch.cumsum(wm, -1)
    W_ex, WM_ex = W_in - w, WM_in - wm
    W_suf, WM_suf = W_in[:, -1:] - W_in, WM_in[:, -1:] - WM_in
    return 2.0 * (mid * W_ex - WM_ex + WM_suf - mid * W_suf) + (2.0 / 3.0) * w * width


def fp32_bounds(sigma, z, rays_d, near, far, g_loss, C=8.0):
    """the tolerance of the fp32 kernels, element by element: C * 2^-24 times the sensitivity of each result to one
    rounding per operation.  The weights carry the arithmetic of b2n_composite_fwd: alpha = 1 - exp(-x) and
    a = 1 - alpha + 1e-10 are rounded in absolute terms, so a factor a_k of the transmittance has a relative error of
    up to 2^-24 (1 + alpha_k / a_k), which is large where alpha_k rounds to 1 (a nearly opaque sample):
    S_i = 1 + sum_{k<i} (1 + alpha_k / a_k) bounds the relative error of T_i in units of 2^-24.  The prefix sums of the
    loss and of dL/dw add N roundings, exp adds |x| (the rounding of its argument x = sigma tau).
      loss:    Wt N + (G + Wt) sum_i w_i S_i
      g_sigma: tau_i (G + Wt) |g_loss| (e_i T_i (S_i + |x_i| + N) + sum_{j>i} w_j (S_j + N)),
    G = max |dL/dw|, Wt = sum w; the second term is the error of the reverse scan R_i (e_i / a_i <= 1).
    Returns (loss bound [B], g_sigma bound [B,N])."""
    sigma, z, rays_d = sigma.double(), z.double(), rays_d.double()
    B, N = z.shape
    eps = 2.0 ** -24
    dn = rays_d.norm(dim=-1)
    tau = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1) * dn[:, None]
    x = sigma * tau
    e = torch.exp(-x)
    alpha = 1.0 - e
    a = 1.0 - alpha + 1e-10
    T = torch.cumprod(torch.cat([torch.ones_like(a[:, :1]), a[:, :-1]], -1), -1)
    w = alpha * T
    mid, width = intervals(z, float(near), float(far))
    Wt = w.sum(-1, keepdim=True)
    G = grad_w(w, mid, width).abs().amax(-1, keepdim=True)
    per = 1.0 + alpha / a
    S = 1.0 + torch.cumsum(per, -1) - per                               # 1 + sum_{k<i}
    wS = w * (S + N)
    after = (wS.sum(-1, keepdim=True) - torch.cumsum(wS, -1)).clamp_min(0.0)   # sum_{j>i}
    gb = C * eps * tau * (G + Wt) * g_loss.double().abs()[:, None] * (e * T * (S + x.abs() + N) + after) + 1e-30
    lb = C * eps * (N * Wt[:, 0] + (G + Wt)[:, 0] * (w * S).sum(-1)) + 1e-30
    return lb, gb
