"""Renderer of the hot path on B200 kernels (reference src/renderer.py).

DensityGrid        <- reference :5-183   (bool + fp32 buffers kept for the API / checkpoints,
                                          a packed bitfield is what the kernels read)
sample_stratified  <- reference :186-201
volume_render      <- reference :204-237
render_rays        <- reference :240-384  (march -> compact -> model -> composite; ONE host sync
                                          instead of three, no scatter-into-zeros pass)
render_image       <- reference :387-418
"""
import numpy as np
import torch
from torch import nn

import b2n
from b2n import march as _march
from b2n._lib import call, ptr, require_cuda, stream


class DensityGrid(nn.Module):
    def __init__(self, resolution=128, bound=1.0, threshold=0.01):
        super().__init__()
        self.resolution, self.bound, self.threshold = resolution, bound, threshold
        self.register_buffer("grid", torch.zeros(resolution, resolution, resolution))
        self.register_buffer("binary_grid", torch.ones(resolution, resolution, resolution, dtype=torch.bool))
        self.scale = resolution / (2 * bound)
        self.offset = bound
        self._bits = None
        self._bits_key = None

    # the kernels read a bitfield; rebuild it whenever binary_grid was replaced or written
    def bits(self):
        """The cache is keyed on the tensor OBJECT (a weak reference: a re-assigned ``binary_grid`` is a different
        object even when the allocator hands it the freed block of the old one at version 0), its storage pointer and
        its in-place version counter."""
        import weakref
        bg = self.binary_grid
        key = (bg.data_ptr(), bg._version, str(bg.device))
        owner = self._bits_owner() if getattr(self, "_bits_owner", None) is not None else None
        if self._bits is None or self._bits_key != key or owner is not bg:
            self._bits = _march.pack_occupancy(bg)
            self._bits_key = key
            self._bits_owner = weakref.ref(bg)
        return self._bits

    def _lattice(self, device):
        """the R^3 corner lattice of ``update`` (reference :49-54), built once per device"""
        key = (str(torch.device(device)), self.resolution, float(self.bound))
        if getattr(self, "_lattice_key", None) != key:
            ax = torch.linspace(-self.bound, self.bound, self.resolution, device=device)
            self._lattice_pts = torch.stack(torch.meshgrid(ax, ax, ax, indexing="ij"), dim=-1).reshape(-1, 3).contiguous()
            self._lattice_key = key
        return self._lattice_pts

    @torch.no_grad()
    def update(self, model, n_samples=128 ** 3, device="cuda", time=None, decay=1.0, **_unused):
        """Re-evaluate sigma on the R^3 corner lattice and refresh grid / binary_grid.
        Accepts (and ignores) the extra keywords run.py:1982-1985 passes.  A model that offers ``density(x, t=None)``
        (this package's NeuralField) is swept through it -- sigma only, no colour branch (SURVEY 8f-3); any other
        model is called like the reference does, with zero view directions."""
        R = self.resolution
        pts = self._lattice(device)
        mode = getattr(model, "mode", "unknown")
        # The reference sweeps the lattice in 2^18-point batches (a memory limit of its hardware, :73-80) and, for Part 4,
        # once per time anchor (:65-86).  Every kernel here is per-point, so the batch size does not change a single bit
        # of sigma: the sweep runs in calls of up to 2^21 points, and Part 4's three anchors ride in ONE pass (points
        # repeated per anchor, each with its own time) followed by the max over the anchors.
        batch = 2 ** 21
        density = getattr(model, "density", None)
        n = pts.shape[0]

        def sweep(times):
            """sigma [len(times), n]: one (batched) evaluation per time value (None: static model)"""
            k = len(times)
            out = torch.empty(k, n, device=pts.device)
            flat = out.view(-1)
            if times[0] is not None:
                tcol = torch.cat([tv.to(pts.device, torch.float32).reshape(1, 1).expand(n, 1) for tv in times])
            for i in range(0, k * n, batch):
                j = min(i + batch, k * n)
                if k == 1 or (i // n == (j - 1) // n):                # inside one anchor: a view of the lattice
                    p = pts[i % n:(j - 1) % n + 1]
                else:                                                  # spans anchors: gather the wrapped range
                    p = pts[torch.arange(i, j, device=pts.device) % n]
                tt = None if times[0] is None else tcol[i:j]
                if density is not None:
                    s = density(p) if tt is None else density(p, t=tt)
                elif tt is None:
                    _, s = model(p, torch.zeros_like(p))
                else:
                    _, s, _ = model(p, torch.zeros_like(p), t=tt)
                flat[i:j] = s.reshape(-1)
            return out

        if mode == "part4":
            # run.py:1972-1986 calls update() three times in a row with different ``time`` arguments, which Part 4
            # ignores (reference :65-86): the three sweeps see the same model and return the same sigma.  The sweep is
            # re-used while no parameter of the model has changed (autograd's version counters, which every in-place
            # optimizer update bumps -- b2n.optim.FusedAdamW included); decay / threshold are applied per call below
            key = (tuple((id(p), p._version) for p in model.parameters()), bool(getattr(model, "training", False)),
                   str(pts.device), R, float(self.bound))
            cached = getattr(self, "_sweep_cache", None)
            if cached is not None and cached[0] == key:
                cur = cached[1]
            else:
                cur = sweep([torch.tensor(a) for a in (0.0, 0.5, 1.0)]).amax(dim=0)
                self._sweep_cache = (key, cur)
        elif mode == "part3":
            if time is None:
                raise ValueError("Part 3 density grid update requires a time parameter")
            cur = sweep([time.reshape(-1)[0]])[0]
        else:
            cur = sweep([None])[0]
        cur = cur.contiguous()
        # every buffer the kernel touches lives on the device of the sweep (the registered buffers may still sit on
        # the CPU or on another GPU when the caller never moved the grid: the reference simply rebinds them, :122-128)
        if mode in ("part3", "part4"):
            grid = self.grid.to(cur.device, torch.float32).contiguous().clone()
        else:
            grid = torch.empty(R, R, R, device=cur.device)
        require_cuda(cur, grid)
        binary = torch.empty(R, R, R, device=cur.device, dtype=torch.bool)
        bits = torch.empty((R ** 3 + 31) // 32, device=cur.device, dtype=torch.int32)
        n_active = torch.empty(1, device=cur.device, dtype=torch.int64)
        call("b2n_occ_update", ptr(cur), ptr(grid), R ** 3, int(mode in ("part3", "part4")), float(decay),
             float(self.threshold), ptr(binary.view(torch.uint8)), ptr(bits), ptr(n_active), stream())
        self.grid = grid
        self.binary_grid = binary
        import weakref
        self._bits, self._bits_key = bits, (binary.data_ptr(), binary._version, str(binary.device))
        self._bits_owner = weakref.ref(self.binary_grid)
        # binary.float().mean(): fp32 mean of 0/1 values, then .item()
        ratio = float(np.float32(n_active.item()) / np.float32(R ** 3))
        b2n.check_errors()                     # a host sync just happened: look at every outstanding tcgen05 abort flag
        return ratio

    def get_active_mask(self, pts):
        return _march.active_mask(pts, self.bits(), self.resolution, self.bound)

    def should_update(self, step, update_interval=16, warmup_iters=0):
        return step >= warmup_iters and step % update_interval == 0


def sample_stratified(near, far, n_samples, n_rays, device, perturb):
    """Depths [n_rays, n_samples]; with ``perturb`` one torch.rand draw of that shape, like the reference."""
    dev = torch.device(device)
    u = torch.rand((n_rays, n_samples), device=dev) if perturb else None
    dummy = torch.zeros(n_rays, 3, device=dev)
    return _march.march(dummy, dummy, near, far, n_samples, u).z


def volume_render(rgb, sigma, z_vals, rays_d, bg_color=None):
    """rgb [B,N,3], sigma [B,N] -> (rgb_map [B,3], depth_map [B], acc_map [B])."""
    color, depth, acc, _ = b2n.composite(rgb, sigma, z_vals, rays_d, bg=bg_color)
    return color, depth, acc


def render_rays(model, rays_o, rays_d, near, far, n_samples, perturb, density_grid=None, times=None,
                white_bkgd=True, bg_color=None, _jitter=None):
    """``_jitter`` (private, tests only): a [n_rays, n_samples] U[0,1) tensor to use instead of drawing
    ``torch.rand`` -- lets parity tests feed the very jitter the CPU reference drew."""
    color, depth, acc, extras, _ = b2n.render.render_rays_train(
        model, rays_o, rays_d, near, far, n_samples, perturb, density_grid=density_grid, times=times,
        white_bkgd=white_bkgd, bg_color=bg_color, _jitter=_jitter)
    if times is None:
        return color, depth, acc
    return color, depth, acc, extras


def render_image(model, rays_o, rays_d, near, far, n_samples, chunk, white_bkgd):
    h, w = rays_o.shape[:2]
    rays_o, rays_d = rays_o.reshape(-1, 3), rays_d.reshape(-1, 3)
    out = torch.empty(rays_o.shape[0], 3, device=rays_o.device)
    for i in range(0, rays_o.shape[0], chunk):
        out[i:i + chunk] = render_rays(model=model, rays_o=rays_o[i:i + chunk], rays_d=rays_d[i:i + chunk],
                                       near=near, far=far, n_samples=n_samples, perturb=False,
                                       white_bkgd=white_bkgd)[0]
    if not torch.cuda.is_current_stream_capturing():
        b2n.check_errors()                     # the image is about to be read by the caller: no silent garbage
    return out.view(h, w, 3)
