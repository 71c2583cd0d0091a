"""float64 restatement of the pose-refinement contract (b2n.PoseRefinement, b2n_sample_rays_bwd and
b2n_march_points_bwd of include/b2nerf.h, DESIGN.md §5k): the corrected poses, the rays of pixel picks, the sample
points o + d z, and the gradient w.r.t. the corrections xi by autograd.  The view direction the decoders see is a
constant (detached), and |d| enters nothing else.  Device-agnostic torch; written apart from b2n/pose.py."""
import numpy as np
import torch


def exp_so3(omega):
    """Rodrigues in float64, [..., 3] -> [..., 3, 3]; the Taylor series below theta^2 = 1e-12"""
    omega = omega.double()
    th2 = (omega ** 2).sum(-1, keepdim=True)[..., None]
    small = th2 < 1e-12
    th = torch.sqrt(torch.where(small, torch.ones_like(th2), th2))
    A = torch.where(small, 1 - th2 / 6 + th2 ** 2 / 120, torch.sin(th) / th)
    B = torch.where(small, 0.5 - th2 / 24 + th2 ** 2 / 720, (1 - torch.cos(th)) / torch.where(small, 1.0, th2))
    K = torch.zeros(*omega.shape[:-1], 3, 3, dtype=torch.float64, device=omega.device)
    K[..., 0, 1], K[..., 0, 2], K[..., 1, 2] = -omega[..., 2], omega[..., 1], -omega[..., 0]
    K = K - K.transpose(-1, -2)
    eye = torch.eye(3, dtype=torch.float64, device=omega.device)
    return eye + A * K + B * (K @ K)


def corrected(poses, xi):
    """[V,4,4] poses, xi [V,6] = (omega, rho) -> c2w [[exp(omega), rho], [0, 1]] (float64)"""
    poses, xi = poses.double(), xi.double()
    R, t = poses[:, :3, :3], poses[:, :3, 3]
    R2 = R @ exp_so3(xi[:, :3])
    t2 = (R @ xi[:, 3:, None])[..., 0] + t
    out = poses.clone()
    out[:, :3, :3], out[:, :3, 3] = R2, t2
    return out


def cam_dirs(pix_y, pix_x, H, W, focal):
    """the sampler's camera direction, with the fp32 roundings of b2n_sample_rays: ((x - W/2)/f, -(y - H/2)/f, -1)"""
    f = np.float32(focal)
    x = pix_x.cpu().numpy().astype(np.float32)
    y = pix_y.cpu().numpy().astype(np.float32)
    cx = (x - np.float32(W * 0.5)) / f
    cy = -((y - np.float32(H * 0.5)) / f)
    c = np.stack([cx, cy, -np.ones_like(cx)], -1).astype(np.float64)
    return torch.from_numpy(c)


def rays(c2w, img_idx, pix_y, pix_x, H, W, focal, scene_scale):
    """(rays_o, rays_d) [B,3] float64 of the picks under poses c2w [V,4,4] (differentiable w.r.t. c2w)"""
    c = cam_dirs(pix_y, pix_x, H, W, focal).to(c2w.device)
    M = c2w[img_idx.to(c2w.device)]
    d = (M[:, :3, :3] @ c[..., None])[..., 0]
    return M[:, :3, 3] * scene_scale, d / d.norm(dim=-1, keepdim=True)


def points(rays_o, rays_d, z):
    """o + d z: [B,N,3]"""
    return rays_o[:, None, :] + rays_d[:, None, :] * z.double()[..., None]


def points_bwd(z, g_pts):
    """(g_o, g_d) [B,3] of dense g_pts [B,N,3] (inactive samples: 0) in float64"""
    g = g_pts.double()
    return g.sum(1), (z.double()[..., None] * g).sum(1)


def rays_bwd(poses, img_idx, pix_y, pix_x, H, W, focal, scene_scale, g_o, g_d):
    """g_poses [V,4,4] of sum(g_o . rays_o + g_d . rays_d) by autograd (float64)"""
    P = poses.detach().double().requires_grad_(True)
    o, d = rays(P, img_idx, pix_y, pix_x, H, W, focal, scene_scale)
    L = (o * g_o.double()).sum() + (d * g_d.double()).sum()
    (g,) = torch.autograd.grad(L, P)
    g = g.clone()
    g[:, 3, :] = 0.0
    return g


def xi_grad(poses, xi, picks, H, W, focal, scene_scale, z, g_pts):
    """g_xi [V,6] of sum(g_pts . (o + d z)) through the corrected poses (float64, autograd)"""
    x = xi.detach().double().requires_grad_(True)
    o, d = rays(corrected(poses, x), *picks, H, W, focal, scene_scale)
    L = (points(o, d, z) * g_pts.double()).sum()
    (g,) = torch.autograd.grad(L, x)
    return g
