#!/usr/bin/env python
"""Timings of camera pose refinement (b2n.PoseRefinement, DESIGN.md §5k) at C2 size -- development aid.

    python tools/pose_bench.py [--iters 50] [--steps 20]

1. b2n_march_points_bwd alone with CUDA events: B = 2^18 rays x N = 128 samples, dense and compacted by the ball
   occupancy of synthetic.ball_occupancy, against the bytes it must move at 7.7 TB/s.
2. b2n_sample_rays_bwd alone: 2^18 rays over V = 100 views.
3. A C2-configured training step (bench.py's model, optimiser, TV term and gradient clipping; ball occupancy, then
   dense without a grid, where the hash grid runs in spatial order) on rays of 100 resident views of 800^2, without and with pose refinement, alternated in the same process; then one step of
   each leg under b2n's per-entry-point profiler for the split (the hash grid loses its spatial order when its input
   needs a gradient, and its backward gains the input gradient).
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "project-nerf_b200")]
import numpy as np  # noqa: E402
import torch  # noqa: E402

import b2n  # noqa: E402
from b2n import _lib, errormap, march, synthetic  # noqa: E402

C2 = dict(mode="part2_instant", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
          per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
NEAR, FAR, N, B, GRID_R, V, HW = 2.0, 6.0, 128, 2 ** 18, 128, 100, 800
HBM_BYTES_PER_S = 7.7e12           # HGX B200 data sheet, one GPU


def events(fn, iters, warm):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def report(name, t, best, nbytes):
    bound_us = nbytes / HBM_BYTES_PER_S * 1e6
    print(f"{name:52s}: median {t * 1e3:8.1f} us  best {best * 1e3:8.1f} us  bytes {nbytes / 1e6:7.1f} MB -> "
          f"bound {bound_us:6.1f} us = {100 * bound_us / (t * 1e3):5.1f} % of the median", flush=True)


def bench_points(args):
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(B, seed=1))
    u = torch.rand(B, N, device="cuda")
    bits = march.pack_occupancy(synthetic.ball_occupancy(GRID_R, 1.5).cuda())
    for name, kw in (("dense", {}), ("ball occupancy, compact", dict(bits=bits, R=GRID_R, bound=1.5))):
        m = march.march(ro, rd, NEAR, FAR, N, u, **kw)
        P = m.n_active
        g_pts = torch.randn(P, 3, device="cuda")
        g_o, g_d = torch.empty(B, 3, device="cuda"), torch.empty(B, 3, device="cuda")

        def run():
            _lib.call("b2n_march_points_bwd", _lib.ptr(m.z), _lib.ptr(m.mask_words), _lib.ptr(m.ray_offset),
                      _lib.ptr(g_pts), B, N, _lib.ptr(g_o), _lib.ptr(g_d), _lib.stream())

        t, best = events(run, args.iters, args.warmup)
        layout = (4 * ((N + 31) // 32) + 4) * B if m.mask_words is not None else 0
        nbytes = 12 * P + 4 * B * N + layout + 24 * B          # g_pts, the rays' z, the layout, g_o + g_d
        report(f"march_points_bwd {name} (P={P})", t, best, nbytes)


def bench_rays_bwd(args):
    poses = synthetic.hemisphere_poses(V, seed=0).cuda()
    picks = tuple(torch.randint(0, n, (B,), device="cuda") for n in (V, HW, HW))
    g_o, g_d = torch.randn(B, 3, device="cuda"), torch.randn(B, 3, device="cuda")
    g_poses = torch.empty(V, 4, 4, device="cuda")
    scratch = torch.empty(int(_lib.lib.b2n_sample_rays_bwd_scratch(B, V)), dtype=torch.uint8, device="cuda")
    focal = float(np.float32(0.5 * HW / np.tan(0.5 * synthetic.CAMERA_ANGLE_X)))

    def run():
        _lib.call("b2n_sample_rays_bwd", _lib.ptr(poses), *(_lib.ptr(t) for t in picks), B, V, HW, HW, focal, 1.0,
                  _lib.ptr(g_o), _lib.ptr(g_d), _lib.ptr(g_poses), _lib.ptr(scratch), _lib.stream())

    t, best = events(run, args.iters, args.warmup)
    nbytes = B * (3 * 8 + 24 + 24) + 2 * B * 8 + 64 * V     # picks, g_o, g_d; the sort's keys and values; g_poses
    report(f"sample_rays_bwd B=2^18 V={V}", t, best, nbytes)


def _dataset():
    from src.dataset import BlenderDataset

    class Resident(BlenderDataset):
        """100 random 800^2 views held in memory: the resident copies are all the sampler reads"""

        def __init__(self):
            self._dev = {}
            self.poses = synthetic.hemisphere_poses(V, seed=0)
            self._rgba8 = np.random.RandomState(0).randint(0, 256, (V, HW, HW, 4), dtype=np.uint8)
            self.H = self.W = HW
            self.focal = 0.5 * HW / np.tan(0.5 * synthetic.CAMERA_ANGLE_X)
            self.scene_scale, self.white_bkgd, self._images = 1.0, True, None

    return Resident()


def bench_step(args, with_grid):
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    torch.manual_seed(0)
    dev = "cuda"
    ds = _dataset()
    model = NeuralField(C2).to(dev).train()
    refine = b2n.PoseRefinement(V)
    table = model.representation.encoding.params
    opt = torch.optim.AdamW(model.parameters(), lr=0.01, weight_decay=1e-5)
    opt_pose = torch.optim.Adam(refine.parameters(), lr=1e-4)
    grid = DensityGrid(resolution=GRID_R, bound=1.5, threshold=0.12).to(dev)
    grid.binary_grid = synthetic.ball_occupancy(GRID_R, 1.5).to(dev)
    bg = torch.ones(3, device=dev)
    gen = torch.Generator(device=dev).manual_seed(1)

    def step(with_pose):
        picks = tuple(torch.randint(0, n, (B,), device=dev, generator=gen) for n in (V, HW, HW))
        ro, rd, rgba = refine.rays(ds, picks) if with_pose else errormap.rays(ds, picks)
        target = rgba[:, :3] * rgba[:, 3:4] + bg * (1.0 - rgba[:, 3:4])
        pred, _, _ = render_rays(model, ro, rd, NEAR, FAR, N, True, density_grid=grid if with_grid else None,
                                 bg_color=bg)
        loss = torch.nn.functional.mse_loss(pred, target)
        loss = loss + torch.mean(torch.abs(table[1:] - table[:-1])) * 1e-6
        opt.zero_grad(set_to_none=False)
        opt_pose.zero_grad(set_to_none=False)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.representation.parameters(), max_norm=1.0)
        torch.nn.utils.clip_grad_norm_(model.decoder.parameters(), max_norm=1.0)
        opt.step()
        if with_pose:
            opt_pose.step()

    for _ in range(args.warmup):
        step(False)
        step(True)
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for i in range(args.steps):
        for with_pose in ((False, True) if i % 2 == 0 else (True, False)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(with_pose)
            e1.record()
            torch.cuda.synchronize()
            times[with_pose].append(e0.elapsed_time(e1))
    b2n.check_errors()
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    occ = "ball occupancy" if with_grid else "dense, no grid"
    print(f"C2 training step (B={B}, N={N}, {occ}, {V} views of {HW}^2), {args.steps} alternated steps each: "
          f"without refinement median {med[False]:.3f} ms, with median {med[True]:.3f} ms "
          f"(+{med[True] - med[False]:.3f} ms, {100 * (med[True] / med[False] - 1):+.2f} %)", flush=True)
    # the split: one profiled step of each leg (events around every C-ABI call; slower than the timed steps)
    split = {}
    for with_pose in (False, True):
        acc = {}
        for _ in range(3):
            _lib.PROFILER = _lib.Profiler()
            step(with_pose)
            torch.cuda.synchronize()
            for k, v in _lib.PROFILER.summary().items():
                acc.setdefault(k, []).append(v["ms"])
            _lib.PROFILER = None
        split[with_pose] = {k: sorted(v)[len(v) // 2] for k, v in acc.items()}
    for k in sorted(set(split[False]) | set(split[True])):
        a, b = split[False].get(k, 0.0), split[True].get(k, 0.0)
        if abs(b - a) >= 0.005 or k in ("b2n_hash_fwd", "b2n_hash_bwd", "b2n_hash_order"):
            print(f"  split {k:28s}: without {a:7.3f} ms  with {b:7.3f} ms  ({b - a:+.3f} ms)", flush=True)
    tot = {k: sum(v.values()) for k, v in split.items()}
    print(f"  split sum of all entry points: without {tot[False]:.3f} ms  with {tot[True]:.3f} ms "
          f"({tot[True] - tot[False]:+.3f} ms); the rest of the step difference is torch work (the V-sized pose "
          f"composition and its backward, the pose optimiser)", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("pose_bench needs a CUDA device")
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, power.max_limit: {smi}", flush=True)
    bench_points(args)
    bench_rays_bwd(args)
    bench_step(args, with_grid=True)
    bench_step(args, with_grid=False)


if __name__ == "__main__":
    main()
