"""Error-map ray sampling: draw training pixels in proportion to a per-view map of recent loss, mixed with a uniform
share, as Instant-NGP does (b2n_errormap_* of include/b2nerf.h; the contract is documented there and in DESIGN.md §5i).

    emap = ErrorMap(len(dataset), dataset.H, dataset.W)
    picks, ratio = emap.sample(batch_size)                       # every step
    rays_o, rays_d, target = rays(dataset, picks)                # what sample_random_rays returns for these picks
    ...
    emap.update(picks, ((pred - target[:, :3]) ** 2).mean(-1).detach())

``sample`` and ``update`` run on the GPU without a host synchronisation (both can be captured in a CUDA graph), use no
float atomics and give the same bits on every run.  The reference draws its rays uniformly; ``sample_random_rays`` is
unchanged and this is a separate sampler, off unless asked for.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from ._lib import call, lib, ptr, require_cuda, stream

DEFAULT_CELLS = (128, 128)


def _int(name, v, lo, hi=None):
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)) or v < lo or (hi is not None and v > hi):
        rng = f"[{lo}, {hi}]" if hi is not None else f">= {lo}"
        raise ValueError(f"{name} must be an int in {rng}, got {v!r}")
    return int(v)


def _frac(name, v):
    if isinstance(v, bool) or not isinstance(v, (int, float, np.integer, np.floating)) or not 0.0 <= float(v) <= 1.0:
        raise ValueError(f"{name} must be a number in [0, 1], got {v!r}")
    return float(v)


def _check_picks(picks, B=None):
    """picks = (img_idx, pix_y, pix_x): three int64 CUDA tensors of one shape [B]"""
    if not isinstance(picks, (tuple, list)) or len(picks) != 3 or not all(isinstance(t, torch.Tensor) for t in picks):
        raise ValueError("picks must be a tuple (img_idx, pix_y, pix_x) of tensors")
    require_cuda(*picks)
    shape = picks[0].shape
    if len(shape) != 1 or any(t.shape != shape for t in picks) or any(t.dtype != torch.int64 for t in picks):
        raise ValueError(f"picks must be three int64 [B] tensors, got {[(tuple(t.shape), t.dtype) for t in picks]}")
    if B is not None and shape[0] != B:
        raise ValueError(f"picks hold {shape[0]} rays, expected {B}")
    return tuple(t.contiguous() for t in picks)


class ErrorMap:
    """A map ``e [V, Hm, Wm]`` (fp32, -1 = never observed) of the recent per-pixel error of V views of H x W pixels,
    with its integer accumulators and the fp64 CDF over its cells.

    ``cells`` = (Hm, Wm), clipped to (H, W); ``beta``: the momentum of the update; ``uniform_frac``: the share of rays
    drawn uniformly over all pixels (λ).  Pixel (y, x) lies in cell (floor(y Hm / H), floor(x Wm / W))."""

    def __init__(self, n_views, H, W, cells=DEFAULT_CELLS, beta=0.1, uniform_frac=0.25, device="cuda"):
        self.V = _int("n_views", n_views, 1)
        self.H, self.W = _int("H", H, 1), _int("W", W, 1)
        if not isinstance(cells, (tuple, list)) or len(cells) != 2:
            raise ValueError(f"cells must be a pair (Hm, Wm), got {cells!r}")
        self.Hm = min(_int("cells[0]", cells[0], 1), self.H)
        self.Wm = min(_int("cells[1]", cells[1], 1), self.W)
        if self.V * self.Hm * self.Wm >= 2 ** 31:
            raise ValueError(f"need n_views * Hm * Wm < 2^31, got {self.V} * {self.Hm} * {self.Wm}")
        self.beta = _frac("beta", beta)
        self.uniform_frac = _frac("uniform_frac", uniform_frac)
        dev = torch.device(device)
        if dev.type != "cuda":
            raise ValueError("ErrorMap needs a CUDA device: this package has no CPU path for the error-map sampler")
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        self.device = dev
        n = self.V * self.Hm * self.Wm
        self.e = torch.full((self.V, self.Hm, self.Wm), -1.0, device=dev)
        self.acc_sum = torch.zeros(n, dtype=torch.int64, device=dev)       # uint64 bits (values < 2^63)
        self.acc_cnt = torch.zeros(n, dtype=torch.int32, device=dev)       # uint32 bits (values < 2^31)
        self.cdf = torch.zeros(n, dtype=torch.float64, device=dev)         # the CDF of the all-unobserved map
        self._scratch = torch.empty(int(lib.b2n_errormap_scratch(self.V, self.Hm, self.Wm)), dtype=torch.uint8,
                                    device=dev)

    @property
    def shape(self):
        return self.V, self.H, self.W

    def sample(self, batch_size, generator: Optional[torch.Generator] = None, u: Optional[torch.Tensor] = None
               ) -> Tuple[Tuple[torch.Tensor, torch.Tensor, torch.Tensor], torch.Tensor]:
        """``batch_size`` pixel picks ((img_idx, pix_y, pix_x) int64 [B]) and ``ratio`` [B] fp32 = 1 / (V H W p(pick)),
        the weight that makes a per-ray loss unbiased when uniform_frac > 0 (returned only, never applied).  The
        uniforms ``u`` [B,3] are ``torch.rand`` on the map's device (with ``generator`` if given) unless passed in."""
        B = _int("batch_size", batch_size, 0)
        if u is None:
            u = torch.rand((B, 3), device=self.device, generator=generator)
        else:
            if not isinstance(u, torch.Tensor) or u.shape != (B, 3):
                raise ValueError(f"u must be a [batch_size, 3] tensor, got {getattr(u, 'shape', u)}")
            require_cuda(u)
            if u.device != self.device:
                raise ValueError(f"u lives on {u.device}, the map on {self.device}")
            u = u.detach().float().contiguous()
        img_idx, pix_y, pix_x = (torch.empty(B, dtype=torch.int64, device=self.device) for _ in range(3))
        ratio = torch.empty(B, device=self.device)
        with torch.cuda.device(self.device):
            call("b2n_errormap_sample", ptr(self.e), ptr(self.cdf), ptr(u), B, self.V, self.H, self.W, self.Hm,
                 self.Wm, self.uniform_frac, ptr(img_idx), ptr(pix_y), ptr(pix_x), ptr(ratio), stream(),
                 work=(B * (12.0 + 8.0 * 22 + 4.0 + 28.0), 0.0))
        return (img_idx, pix_y, pix_x), ratio

    def update(self, picks, err: torch.Tensor, group=None) -> None:
        """Fold the per-ray errors ``err`` [B] (e.g. the detached per-ray MSE) of the rays ``picks`` into the map and
        rebuild the CDF.  ``group``: a ``torch.distributed`` process group whose ranks each pass their own picks;
        the integer accumulators are all-reduced (SUM) before they are applied, so every rank ends with the map of the
        concatenated batch, bit for bit."""
        if not isinstance(err, torch.Tensor) or err.dim() != 1:
            raise ValueError(f"err must be a [B] tensor, got {getattr(err, 'shape', err)}")
        picks = _check_picks(picks, err.shape[0])
        require_cuda(err, *picks)
        if err.device != self.device:
            raise ValueError(f"err lives on {err.device}, the map on {self.device}")
        B = err.shape[0]
        world = 1
        if group is not None:
            import torch.distributed as dist
            world = dist.get_world_size(group)
        if B * world >= 2 ** 31:
            raise ValueError(f"an update takes fewer than 2^31 rays over all ranks, got {B} x {world}")
        err = err.detach().float().contiguous()
        with torch.cuda.device(self.device):
            call("b2n_errormap_accumulate", *(ptr(t) for t in picks), ptr(err), B, self.V, self.H, self.W, self.Hm,
                 self.Wm, ptr(self.acc_sum), ptr(self.acc_cnt), stream(), work=(B * 40.0, 0.0))
            if group is not None:
                import torch.distributed as dist
                dist.all_reduce(self.acc_sum, op=dist.ReduceOp.SUM, group=group)
                dist.all_reduce(self.acc_cnt, op=dist.ReduceOp.SUM, group=group)
            n = self.acc_cnt.numel()
            call("b2n_errormap_apply", ptr(self.e), ptr(self.acc_sum), ptr(self.acc_cnt), self.V, self.Hm, self.Wm,
                 self.beta, stream(), work=(n * 16.0, 0.0))
            self.rebuild_cdf()

    def rebuild_cdf(self) -> None:
        """rebuild the CDF from ``e`` (``update`` does it; call it after writing ``e`` directly)"""
        n = self.cdf.numel()
        with torch.cuda.device(self.device):
            call("b2n_errormap_cdf", ptr(self.e), self.V, self.Hm, self.Wm, ptr(self.cdf), ptr(self._scratch),
                 stream(), work=(n * 16.0, 0.0))

    def rays(self, dataset, picks):
        """``rays(dataset, picks)`` for a dataset of this map's shape"""
        if (len(dataset), dataset.H, dataset.W) != self.shape:
            raise ValueError(f"the dataset holds {len(dataset)} views of {dataset.H} x {dataset.W}, the map "
                             f"{self.V} of {self.H} x {self.W}")
        return rays(dataset, picks)


def rays(dataset, picks):
    """Exactly what ``dataset.sample_random_rays`` returns for the pixel picks ``picks`` = (img_idx, pix_y, pix_x)
    (int64 CUDA [B], in range, e.g. from ``ErrorMap.sample``): (rays_o, rays_d, target), plus times [B,1] for a
    DynamicDataset.  The same b2n_sample_rays call on the dataset's resident copies."""
    picks = _check_picks(picks)
    with_time = dataset._times_tensor() is not None
    out = dataset._sample(picks[0].shape[0], picks[0].device, with_time=with_time, picks=picks)
    return out if with_time else out[:3]
