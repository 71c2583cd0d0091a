"""Camera pose refinement: learn a small correction of every training view's pose from the photometric loss, as
Instant-NGP ("optimize extrinsics") and nerfstudio's camera optimizer do (b2n_sample_rays_bwd and b2n_march_points_bwd
of include/b2nerf.h; the contract is documented there and in DESIGN.md §5k).

    refine = PoseRefinement(len(dataset)).cuda()
    opt = torch.optim.Adam([{"params": model.parameters(), "lr": 1e-2},
                            {"params": refine.parameters(), "lr": 1e-3}])
    rays_o, rays_d, target = refine.rays(dataset, picks)        # picks = (img_idx, pix_y, pix_x), int64 CUDA [B]
    color, depth, acc = render_rays(model, rays_o, rays_d, ...)  # unchanged: the gradient reaches the poses

View v's correction xi_v = (omega_v, rho_v) (``delta[v]``, zero at the start) right-multiplies its camera-to-world
matrix: R' = R exp(omega) (Rodrigues), t' = R rho + t.  At xi = 0 the rays are bit for bit those of
``sample_random_rays`` / ``b2n.errormap.rays`` for the same picks.  The gradient reaches xi through the sample positions
only: the view directions the decoders see are constants.  The reference's poses are fixed; this module is separate
and off unless asked for.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from ._lib import call, lib, ptr, require_cuda, stream
from .errormap import _check_picks

# below this theta^2 the Rodrigues coefficients are their Taylor series: exact I at omega = 0, and no 0/0 in the
# gradient (torch.where does not mask a NaN of the branch it discards, so that branch is fed a safe theta^2)
TAYLOR_THETA2 = 1e-6


def so3_exp(omega: torch.Tensor) -> torch.Tensor:
    """Rodrigues: omega [..., 3] -> rotation [..., 3, 3] = I + A K + B K^2, K = [omega]_x, A = sin(theta)/theta,
    B = (1 - cos(theta))/theta^2 = 2 sin^2(theta/2)/theta^2, from theta^2 = omega . omega.  Exactly I at omega = 0, with a
    finite gradient there."""
    th2 = (omega * omega).sum(-1)
    small = th2 < TAYLOR_THETA2
    safe = torch.where(small, torch.ones_like(th2), th2)
    th = torch.sqrt(safe)
    a = torch.where(small, 1.0 - th2 / 6.0, torch.sin(th) / th)
    half = torch.sin(0.5 * th)
    b = torch.where(small, 0.5 - th2 / 24.0, 2.0 * half * half / safe)
    x, y, z = omega.unbind(-1)
    zero = torch.zeros_like(x)
    K = torch.stack([zero, -z, y, z, zero, -x, -y, x, zero], -1).reshape(*omega.shape[:-1], 3, 3)
    K2 = (K.unsqueeze(-1) * K.unsqueeze(-3)).sum(-2)
    eye = torch.eye(3, dtype=omega.dtype, device=omega.device)
    return eye + a[..., None, None] * K + b[..., None, None] * K2


def compose(poses: torch.Tensor, xi: torch.Tensor) -> torch.Tensor:
    """c2w' = c2w [[exp(omega), rho], [0, 1]] for poses [V,4,4] and xi = (omega, rho) [V,6].  Written with elementwise
    products and sums (no matmul, so no TF32): at xi = 0 every sum is one term plus exact zeros, and c2w' == c2w."""
    R, t = poses[:, :3, :3], poses[:, :3, 3]
    E = so3_exp(xi[:, :3])
    R2 = (R.unsqueeze(-1) * E.unsqueeze(-3)).sum(-2)
    t2 = (R * xi[:, None, 3:]).sum(-1) + t
    top = torch.cat([R2, t2.unsqueeze(-1)], -1)
    return torch.cat([top, poses[:, 3:, :]], 1)


class _PoseRays(torch.autograd.Function):
    """b2n_sample_rays on the corrected poses; backward b2n_sample_rays_bwd (g_poses [V,4,4])"""

    @staticmethod
    def forward(ctx, poses, img_idx, pix_y, pix_x, rgba8, times, H, W, focal, scene_scale):
        B, V = img_idx.shape[0], poses.shape[0]
        dev = poses.device
        poses = poses.detach().float().contiguous()
        rays_o = torch.empty(B, 3, device=dev)
        rays_d = torch.empty(B, 3, device=dev)
        target = torch.empty(B, 4, device=dev)
        t_out = torch.empty(B, 1, device=dev) if times is not None else torch.empty(0, device=dev)
        call("b2n_sample_rays", ptr(poses), ptr(rgba8), ptr(times), ptr(img_idx), ptr(pix_y), ptr(pix_x), B, V, H, W,
             focal, scene_scale, ptr(rays_o), ptr(rays_d), ptr(target), ptr(t_out) if times is not None else None,
             stream(), work=(B * (24.0 + 4.0 + 24.0 + 24.0 + 16.0 + (8.0 if times is not None else 0.0)), 0.0))
        ctx.save_for_backward(poses, img_idx, pix_y, pix_x)
        ctx.cfg = (H, W, focal, scene_scale)
        ctx.mark_non_differentiable(target, t_out)
        return rays_o, rays_d, target, t_out

    @staticmethod
    def backward(ctx, g_o, g_d, g_target, g_t):
        poses, img_idx, pix_y, pix_x = ctx.saved_tensors
        H, W, focal, scene_scale = ctx.cfg
        B, V = img_idx.shape[0], poses.shape[0]
        dev = poses.device
        g_o = torch.zeros(B, 3, device=dev) if g_o is None else g_o.float().contiguous()
        g_d = torch.zeros(B, 3, device=dev) if g_d is None else g_d.float().contiguous()
        g_poses = torch.empty(V, 4, 4, device=dev)
        scratch = torch.empty(int(lib.b2n_sample_rays_bwd_scratch(B, V)), device=dev, dtype=torch.uint8)
        call("b2n_sample_rays_bwd", ptr(poses), ptr(img_idx), ptr(pix_y), ptr(pix_x), B, V, H, W, focal, scene_scale,
             ptr(g_o), ptr(g_d), ptr(g_poses), ptr(scratch), stream(), work=(B * (24.0 + 24.0 + 24.0 + 32.0), 0.0))
        return g_poses, None, None, None, None, None, None, None, None, None


class PoseRefinement(torch.nn.Module):
    """Per-view pose corrections ``delta`` [V,6] = (omega, rho), zeros at the start, for the V views of a training set.

    ``refine``: optional bool [V]; views outside it keep their pose (xi = delta * refine, so their gradient is exactly
    zero).  ``corrected_poses`` composes in torch; ``rays`` / ``image_rays`` run the ray sampler on the corrected poses
    and return rays through which autograd reaches ``delta``."""

    def __init__(self, n_views: int, refine: Optional[torch.Tensor] = None, device="cuda"):
        super().__init__()
        if isinstance(n_views, bool) or not isinstance(n_views, (int, np.integer)) or n_views < 1:
            raise ValueError(f"n_views must be an int >= 1, got {n_views!r}")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError("PoseRefinement needs a CUDA device: this package has no CPU path for pose refinement")
        self.V = int(n_views)
        self.delta = torch.nn.Parameter(torch.zeros(self.V, 6, device=dev))
        if refine is not None:
            if not isinstance(refine, torch.Tensor) or refine.dtype != torch.bool or refine.shape != (self.V,):
                raise ValueError(f"refine must be a bool tensor of shape ({self.V},), got "
                                 f"{getattr(refine, 'dtype', type(refine))} {tuple(getattr(refine, 'shape', ()))}")
            refine = refine.to(dev)
        self.register_buffer("refine", refine)

    def xi(self) -> torch.Tensor:
        """the corrections in effect, [V,6]: ``delta``, zeroed outside ``refine``"""
        return self.delta if self.refine is None else self.delta * self.refine[:, None].to(self.delta.dtype)

    def corrected_poses(self, poses: torch.Tensor) -> torch.Tensor:
        """poses [V,4,4] -> the corrected camera-to-world matrices [V,4,4], differentiable w.r.t. ``delta``"""
        if not isinstance(poses, torch.Tensor) or poses.shape != (self.V, 4, 4):
            raise ValueError(f"poses must be [{self.V},4,4], got {tuple(getattr(poses, 'shape', ()))}")
        xi = self.xi()
        return compose(poses.to(device=xi.device, dtype=xi.dtype), xi)

    def _check(self, dataset):
        if len(dataset) != self.V:
            raise ValueError(f"the dataset holds {len(dataset)} views, the refinement {self.V}")

    def _rays(self, dataset, img_idx, pix_y, pix_x):
        dev = self.delta.device
        poses, rgba8, times = dataset._resident(dev)
        with torch.cuda.device(dev):
            return _PoseRays.apply(self.corrected_poses(poses), img_idx, pix_y, pix_x, rgba8, times, int(dataset.H),
                                   int(dataset.W), float(np.float32(dataset.focal)), float(dataset.scene_scale))

    def rays(self, dataset, picks):
        """What ``dataset.sample_random_rays`` returns for the pixel picks ``picks`` = (img_idx, pix_y, pix_x) (int64
        CUDA [B], in range, e.g. from ``torch.randint`` or ``ErrorMap.sample``), under the corrected poses: (rays_o,
        rays_d, target), plus times [B,1] for a DynamicDataset.  rays_o and rays_d are differentiable w.r.t. ``delta``."""
        self._check(dataset)
        picks = _check_picks(picks)
        require_cuda(self.delta, *picks)
        rays_o, rays_d, target, t_out = self._rays(dataset, *picks)
        return (rays_o, rays_d, target, t_out) if dataset._times_tensor() is not None else (rays_o, rays_d, target)

    def image_rays(self, dataset, index: int):
        """The rays of every pixel of training view ``index`` under its corrected pose, as ``dataset.get_image_rays``
        lays them out: rays_o, rays_d [H,W,3], the background-composited target [H,W,3] (plus the time [1,1] for a
        DynamicDataset), on the module's device."""
        self._check(dataset)
        if isinstance(index, bool) or not isinstance(index, (int, np.integer)) or not 0 <= index < self.V:
            raise ValueError(f"index must be an int in [0, {self.V}), got {index!r}")
        H, W, dev = int(dataset.H), int(dataset.W), self.delta.device
        y, x = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
        v = torch.full((H * W,), int(index), dtype=torch.int64, device=dev)
        rays_o, rays_d, target, _ = self._rays(dataset, v, y.reshape(-1).contiguous(), x.reshape(-1).contiguous())
        out = (rays_o.view(H, W, 3), rays_d.view(H, W, 3), dataset._composite(target.view(H, W, 4)))
        times = dataset._times_tensor()
        return out + (times[index].view(1, 1).to(dev),) if times is not None else out
