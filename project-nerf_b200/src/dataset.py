"""Blender / D-NeRF dataset loaders with a GPU-resident ray sampler (reference src/dataset.py).

Same classes, constructor arguments, attributes (``poses``, ``images``, ``H``, ``W``, ``focal``,
``camera_angle_x``, ``frames``, ``times``, ``images_rgb``, ``images_alpha``) and methods
(``get_rays``, ``get_image_rays``, ``sample_random_rays``) as the reference, so run.py drives it
unchanged.  Differences are internal:

* the image stack is kept as 8-bit RGBA (lossless for PNG input; the reference's float image is
  ``uint8 / 255``) -- 4x less host memory -- and float views are materialised lazily;
* ``sample_random_rays(batch, device='cuda')`` keeps poses + images in HBM and runs ONE kernel
  (b2n_sample_rays) instead of a CPU gather over a >1 GB float tensor plus three H2D copies.
  The pixel picks are still drawn with the reference's three ``torch.randint`` calls on the CPU
  generator (``rng='cpu'``, default: identical ray selection for identical seeds) or on the device
  generator (``rng='device'``, no host work at all).
"""
import json
import os

import numpy as np
import torch
from PIL import Image


def _load_frames(root_dir, split, downscale):
    with open(os.path.join(root_dir, f"transforms_{split}.json"), "r", encoding="utf-8") as f:
        meta = json.load(f)
    frames = meta["frames"]
    rgba, poses = [], []
    for fr in frames:
        rel = fr["file_path"][2:] if fr["file_path"].startswith("./") else fr["file_path"]
        path = os.path.join(root_dir, rel)
        if not os.path.splitext(path)[1]:
            for ext in (".png", ".jpg"):
                if os.path.exists(path + ext):
                    path += ext
                    break
        img = Image.open(path).convert("RGBA")
        if downscale > 1:
            img = img.resize((img.width // downscale, img.height // downscale), Image.LANCZOS)
        rgba.append(np.asarray(img, dtype=np.uint8))
        poses.append(torch.tensor(fr["transform_matrix"], dtype=torch.float32))
    return meta, frames, np.stack(rgba, axis=0), torch.stack(poses, dim=0)


class BlenderDataset:
    rng = "cpu"          # "cpu": reference-identical pixel picks; "device": draw on the GPU

    def __init__(self, root_dir, split="train", downscale=1, white_bkgd=True, scene_scale=1.0):
        self.root_dir, self.split = root_dir, split
        self.downscale = max(int(downscale), 1)
        self.white_bkgd = white_bkgd
        self.scene_scale = float(scene_scale)
        meta, self.frames, self._rgba8, self.poses = _load_frames(root_dir, split, self.downscale)
        self.camera_angle_x = float(meta["camera_angle_x"])
        self.H, self.W = self._rgba8.shape[1:3]
        self.focal = 0.5 * self.W / np.tan(0.5 * self.camera_angle_x)
        self._directions = self._build_directions()
        self._images = None
        self._dev = {}       # device -> (poses, rgba8[, times]) resident copies
        self._post_init()

    def _post_init(self):
        pass

    # ---- float views of the 8-bit stack (what the reference stores eagerly)
    @property
    def images(self):
        """[N, H, W, 4] float32 RGBA in [0, 1] (CPU)."""
        if self._images is None:
            self._images = torch.from_numpy(self._rgba8.astype(np.float32) / 255.0)
        return self._images

    @images.setter
    def images(self, value):
        """run.py:484 assigns a subset (``val_set.images = test_set.images[val_indices]``): keep the 8-bit
        stack, the float view and the device copies consistent with the assignment."""
        value = value.detach().cpu().float()
        if value.shape[-1] == 4:
            self._rgba8 = (value * 255.0).round().clamp(0, 255).to(torch.uint8).numpy()
        self._images = value
        self._dev = {}

    def _build_directions(self):
        j, i = torch.meshgrid(torch.arange(self.H), torch.arange(self.W), indexing="ij")
        return torch.stack([(i - self.W * 0.5) / self.focal, -(j - self.H * 0.5) / self.focal, -torch.ones_like(i)], dim=-1)

    def __len__(self):
        return self._rgba8.shape[0]

    def get_rays(self, c2w):
        d = self._directions.to(c2w.device).reshape(-1, 3)
        rays_d = torch.matmul(d, c2w[:3, :3].T).reshape(self.H, self.W, 3)
        rays_d = rays_d / torch.norm(rays_d, dim=-1, keepdim=True)
        rays_o = c2w[:3, 3].expand_as(rays_d)
        if self.scene_scale != 1.0:
            rays_o = rays_o * self.scene_scale
        return rays_o, rays_d

    def _composite(self, rgba):
        rgb, alpha = rgba[..., :3], rgba[..., 3:4]
        return rgb * alpha + (1.0 - alpha) if self.white_bkgd else rgb * alpha

    def get_image_rays(self, index, device):
        rays_o, rays_d = self.get_rays(self.poses[index])
        rgba = torch.from_numpy(self._rgba8[index].astype(np.float32) / 255.0)
        return rays_o.to(device), rays_d.to(device), self._composite(rgba).to(device)

    def __setattr__(self, name, value):
        if name == "poses":
            self.__dict__.get("_dev", {}).clear()        # resident copies follow re-assigned poses (run.py:485)
        object.__setattr__(self, name, value)

    # ---- sampling
    def _times_tensor(self):
        return None

    def _resident(self, device):
        key = str(device)
        if key not in self._dev:
            t = self._times_tensor()
            self._dev[key] = (self.poses.to(device).contiguous(), torch.from_numpy(self._rgba8).to(device).contiguous(),
                              t.to(device).contiguous() if t is not None else None)
        return self._dev[key]

    def _draw(self, batch_size, device):
        if self.rng == "device" and torch.device(device).type == "cuda":
            return (torch.randint(0, len(self), (batch_size,), device=device),
                    torch.randint(0, self.H, (batch_size,), device=device),
                    torch.randint(0, self.W, (batch_size,), device=device))
        picks = (torch.randint(0, len(self), (batch_size,)), torch.randint(0, self.H, (batch_size,)),
                 torch.randint(0, self.W, (batch_size,)))
        return picks

    def _sample(self, batch_size, device, with_time, picks=None):
        """rays for ``picks`` = (img_idx, pix_y, pix_x) int64 [batch_size] (in range: b2n_sample_rays does not check
        them), or for a fresh uniform draw when None"""
        img_idx, pix_y, pix_x = self._draw(batch_size, device) if picks is None else picks
        dev = torch.device(device)
        if dev.type == "cuda":
            from b2n._lib import call, ptr, stream
            poses, rgba8, times = self._resident(dev)
            with torch.cuda.device(dev):
                img_idx, pix_y, pix_x = (t.to(dev, non_blocking=True) for t in (img_idx, pix_y, pix_x))
                rays_o = torch.empty(batch_size, 3, device=dev)
                rays_d = torch.empty(batch_size, 3, device=dev)
                target = torch.empty(batch_size, 4, device=dev)
                t_out = torch.empty(batch_size, 1, device=dev) if with_time else None
                call("b2n_sample_rays", ptr(poses), ptr(rgba8), ptr(times), ptr(img_idx), ptr(pix_y), ptr(pix_x),
                     batch_size, len(self), self.H, self.W, float(np.float32(self.focal)), float(self.scene_scale),
                     ptr(rays_o), ptr(rays_d), ptr(target), ptr(t_out), stream())
            return rays_o, rays_d, target, t_out
        raise ValueError("sample_random_rays needs a CUDA device: this package has no CPU path for the training-ray "
                         "sampler (b2n_sample_rays); image-sized host tensors come from get_image_rays")

    def sample_random_rays(self, batch_size, device):
        rays_o, rays_d, target, _ = self._sample(batch_size, device, with_time=False)
        return rays_o, rays_d, target


class DynamicDataset(BlenderDataset):
    """Adds per-frame time stamps (``frame['time']`` or index / (n - 1)); returns RGBA + times."""

    def _post_init(self):
        n = len(self.frames)
        self.times = torch.tensor([fr["time"] if "time" in fr else (i / (n - 1) if n > 1 else 0.0)
                                   for i, fr in enumerate(self.frames)], dtype=torch.float32)
        self._rgb = self._alpha = self._comp = None

    def _times_tensor(self):
        return self.times

    @property
    def images_rgb(self):
        if self._rgb is None:
            self._rgb = BlenderDataset.images.fget(self)[..., :3].contiguous()
        return self._rgb

    @property
    def images_alpha(self):
        if self._alpha is None:
            self._alpha = BlenderDataset.images.fget(self)[..., 3:4].contiguous()
        return self._alpha

    @property
    def images(self):
        """background-composited RGB [N, H, W, 3], like the reference's DynamicDataset.images"""
        if self._comp is None:
            self._comp = self._composite(BlenderDataset.images.fget(self))
        return self._comp

    def get_image_rays(self, index, device):
        rays_o, rays_d = self.get_rays(self.poses[index])
        rgba = torch.from_numpy(self._rgba8[index].astype(np.float32) / 255.0)
        return rays_o.to(device), rays_d.to(device), self._composite(rgba).to(device), self.times[index].view(1, 1).to(device)

    def sample_random_rays(self, batch_size, device):
        return self._sample(batch_size, device, with_time=True)
