#!/usr/bin/env python
"""Timings of the distortion loss (b2n.distortion, DESIGN.md §5j) at C2 size -- development aid.

    python tools/distortion_bench.py [--iters 50] [--steps 20]

1. The op alone, forward and backward, with CUDA events: B = 2^18 rays x N = 128 samples, dense and compacted by the
   ball occupancy of synthetic.ball_occupancy (the sparse leg of bench.py), against the bytes it must move at 7.7 TB/s.
2. A C2-configured training step (bench.py's model, optimiser, TV term and gradient clipping, sparse occupancy) with
   render_rays and with render_rays_distortion + 0.01 * dist.mean(), alternated in the same process.
"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "project-nerf_b200")]
import torch  # noqa: E402

import b2n  # noqa: E402
from b2n import march, synthetic  # noqa: E402

C2 = dict(mode="part2_instant", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
          per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
NEAR, FAR, N, B, GRID_R = 2.0, 6.0, 128, 2 ** 18, 128
HBM_BYTES_PER_S = 7.7e12           # HGX B200 data sheet, one GPU
LAMBDA = 0.01


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


def op_bytes(B, N, P, compact):
    """what each direction must move at least: z and sigma once, rays_d, the layout (mask words + offsets) and the
    per-ray output (forward) or g_loss in and g_sigma out (backward)"""
    layout = (4 * ((N + 31) // 32) + 4) * B if compact else 0
    fwd = 4 * B * N + 4 * P + 12 * B + layout + 4 * B
    bwd = 4 * B * N + 4 * P + 12 * B + layout + 4 * B + 4 * P
    return fwd, bwd


def bench_op(args):
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(B, seed=1))
    u = torch.rand(B, N, device="cuda")
    bits = march.pack_occupancy(synthetic.ball_occupancy(GRID_R, 1.5).cuda())
    for name, kw in (("dense", {}), ("ball occupancy, compact", dict(bits=bits, R=GRID_R, bound=1.5))):
        m = march.march(ro, rd, NEAR, FAR, N, u, **kw)
        P = m.n_active
        sigma = (torch.rand(P, device="cuda") * 4.0).requires_grad_(True)
        g_loss = torch.full((B,), 1.0 / B, device="cuda")
        loss = b2n.distortion(sigma, m.z, rd, NEAR, FAR, m.mask_words, m.ray_offset)

        def fwd():
            b2n.distortion(sigma, m.z, rd, NEAR, FAR, m.mask_words, m.ray_offset)

        def bwd():
            torch.autograd.grad(loss, sigma, g_loss, retain_graph=True)

        tf, tf_best = events(fwd, args.iters, args.warmup)
        tb, tb_best = events(bwd, args.iters, args.warmup)
        bf, bb = op_bytes(B, N, P, m.mask_words is not None)
        for d, t, best, nbytes in (("forward", tf, tf_best, bf), ("backward", tb, tb_best, bb)):
            bound_us = nbytes / HBM_BYTES_PER_S * 1e6
            print(f"op {name:24s} {d:8s}: B={B} N={N} P={P}  median {t * 1e3:8.1f} us  best {best * 1e3:8.1f} us  "
                  f"bytes {nbytes / 1e6:7.1f} MB -> bound {bound_us:6.1f} us = {100 * bound_us / (t * 1e3):5.1f} % of "
                  f"the median", flush=True)


def bench_step(args):
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    torch.manual_seed(0)
    dev = "cuda"
    model = NeuralField(C2).to(dev).train()
    table = model.representation.encoding.params
    opt = torch.optim.AdamW(model.parameters(), lr=0.01, weight_decay=1e-5)
    grid = DensityGrid(resolution=GRID_R, bound=1.5, threshold=0.12).to(dev)
    grid.binary_grid = synthetic.ball_occupancy(GRID_R, 1.5).to(dev)
    bg = torch.ones(3, device=dev)
    batches = [tuple(t.to(dev) for t in synthetic.random_rays(B, seed=i)) for i in range(3)]

    def step(i, with_dist):
        ro, rd, rgba = batches[i % len(batches)]
        target = rgba[:, :3] * rgba[:, 3:4] + bg * (1.0 - rgba[:, 3:4])
        if with_dist:
            pred, _, _, dist = b2n.render_rays_distortion(model, ro, rd, NEAR, FAR, N, True, density_grid=grid,
                                                          bg_color=bg)
            loss = torch.nn.functional.mse_loss(pred, target) + LAMBDA * dist.mean()
        else:
            pred, _, _ = render_rays(model, ro, rd, NEAR, FAR, N, True, density_grid=grid, bg_color=bg)
            loss = torch.nn.functional.mse_loss(pred, target)
        loss = loss + torch.mean(torch.abs(table[1:] - table[:-1])) * 1e-6
        opt.zero_grad(set_to_none=False)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.representation.parameters(), max_norm=1.0)
        torch.nn.utils.clip_grad_norm_(model.decoder.parameters(), max_norm=1.0)
        opt.step()

    for i in range(args.warmup):
        step(i, False)
        step(i, True)
    torch.cuda.synchronize()
    times = {False: [], True: []}
    for i in range(args.steps):
        for with_dist in ((False, True) if i % 2 == 0 else (True, False)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(i, with_dist)
            e1.record()
            torch.cuda.synchronize()
            times[with_dist].append(e0.elapsed_time(e1))
    b2n.check_errors()
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    print(f"C2 training step (B={B}, N={N}, ball occupancy), {args.steps} alternated steps each: without the term "
          f"median {med[False]:.3f} ms, with lambda = {LAMBDA} median {med[True]:.3f} ms "
          f"(+{med[True] - med[False]:.3f} ms, {100 * (med[True] / med[False] - 1):+.2f} %)", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("distortion_bench needs a CUDA device")
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, power.max_limit: {smi}", flush=True)
    bench_op(args)
    bench_step(args)


if __name__ == "__main__":
    main()
