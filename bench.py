#!/usr/bin/env python
"""Throughput benchmark of the ray-marching hot path (contract: see the task brief / DESIGN.md).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1], "C2"): Part 2 Instant-NeRF -- 16-level hash grid (T = 2^19,
F = 2), 64-wide sigma/color MLPs, 128^3 occupancy grid, 2^18 rays per GPU x 128 samples per ray.
A "step" is one full training iteration of run.py:579-630: target compositing, render_rays
(jittered sampling, occupancy test, compaction, hash encode, MLPs, alpha compositing), MSE + TV
loss, backward, gradient all-reduce (N > 1), per-group gradient clipping, AdamW, LR schedule.

Prints ONE JSON line (rank 0).  ``value`` = train rays/s over all GPUs with the ray batches already
resident in HBM; ``e2e`` = the same step fed from pinned HOST buffers (H2D of the batch and D2H of
the loss inside the timed region).  ``--impl reference`` times the reference's CPU implementation
of the same step (the oracle port; the real reference + tcnn shim if /root/reference is present)
on a bounded ray sample.

``--dump-outputs DIR`` (rank 0): after the timed headline steps, what the last of them computed --
rendered color / depth / acc, the loss, and every parameter and its (clipped) gradient after the
optimizer step -- as DIR/<name>.npy in float32.  An array of more than 2^20 elements (the 13 M-entry
hash table and its gradient) is stored as a fixed seeded sample of 2^20 of its elements, so a dump
stays under 64 MB.  Seeds fix every input, so two builds run with the same arguments can be
compared output for output.  The hash-table gradient is summed with atomics and AdamW magnifies
near-zero gradients, so two runs of ONE build already differ.  Two runs of
``python bench.py --no-extras --no-cpu-baseline --dump-outputs DIR`` (the default 20 steps after 3
warm-up steps) on a B200 at its 1000 W power limit differed by relative L2 (||a - b|| / ||b|| per
file) 4e-3 in the hash table, 7e-4 in its gradient, 4e-4 in the decoder weights and 7e-5 in
color / depth / acc.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "project-nerf_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

C2 = dict(mode="part2_instant", n_levels=16, n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
          per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)
NEAR, FAR, N_SAMPLES, GRID_R, GRID_THR = 2.0, 6.0, 128, 128, 0.12
RAYS_PER_GPU = 2 ** 18
LR, WEIGHT_DECAY, ETA_MIN, TV_WEIGHT, TRAIN_ITERS = 0.01, 1e-5, 1e-4, 1e-6, 2000
CPU_SAMPLE_RAYS = 2 ** 14          # BASELINE.md section 2: the CPU arm runs B = 2^14 rays (memory) and says so


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b2n", choices=["b2n", "reference"])
    ap.add_argument("--occupancy", default="dense", choices=["dense", "sparse"])
    ap.add_argument("--rays", type=int, default=RAYS_PER_GPU, help="rays per GPU per step")
    ap.add_argument("--cpu-rays", type=int, default=CPU_SAMPLE_RAYS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sparse-occupancy and render legs")
    ap.add_argument("--only", default=None, help="run only one extra leg (c1_vanilla, c3_dnerf, c4_instant_dnerf, "
                                                 "c5_dualhash) and print its dict -- development aid")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed headline step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b2n" or args.only):
        ap.error("--dump-outputs applies to the headline step of --impl b2n")
    return args


# --------------------------------------------------------------------------------------- CPU arm
def cpu_train_rays_per_s(n_rays, steps, warmup, occupancy):
    """The reference's CPU implementation of the same training step on a bounded ray sample."""
    from oracle import nerf_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    # the reference's own src/: $B2N_REFERENCE, baseline/_ref (git-ignored copy that travels to the GPU box with the
    # snapshot; __graft_entry__.build() refreshes it whenever /root/reference is present), /root/reference
    ref_dir = next((d for d in (os.environ.get("B2N_REFERENCE"), os.path.join(ROOT, "baseline", "_ref"), "/root/reference")
                    if d and os.path.isfile(os.path.join(d, "src", "core.py"))), "")
    occ = torch.ones(GRID_R, GRID_R, GRID_R, dtype=torch.bool) if occupancy == "dense" else O.ball_occupancy(GRID_R, 1.5)
    bg = torch.ones(3)
    kind = "port"
    if os.path.isdir(os.path.join(ref_dir, "src")):
        try:
            from oracle import tcnn_shim
            tcnn_shim.install()
            sys.path.insert(0, ref_dir)
            for m in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
                del sys.modules[m]
            sys.path.remove(PKG)
            from src.core import NeuralField as RefField
            from src import renderer as RefR
            kind = "reference"
        except Exception:
            kind = "port"
    torch.manual_seed(0)
    if kind == "reference":
        model = RefField(C2).train()
        params = list(model.parameters())
        grid = RefR.DensityGrid(resolution=GRID_R, bound=1.5, threshold=GRID_THR)
        grid.binary_grid = occ
        table = model.representation.encoding.params

        def render(ro, rd):
            return RefR.render_rays(model, ro, rd, NEAR, FAR, N_SAMPLES, True, density_grid=grid, bg_color=bg)[0]
    else:
        sd = O.make_state_dict(C2, seed=0)
        sd = {k: (v.requires_grad_(True) if "freq_bands" not in k else v) for k, v in sd.items()}
        params = [v for k, v in sd.items() if v.requires_grad]
        field = O.OracleField(C2, sd)
        table = sd["representation.encoding.params"]

        def render(ro, rd):
            u = torch.rand(ro.shape[0], N_SAMPLES)
            return O.render_rays(field, ro, rd, NEAR, FAR, N_SAMPLES, u, binary_grid=occ, grid_bound=1.5, bg_color=bg)[0]
    opt = torch.optim.AdamW(params, lr=LR, weight_decay=WEIGHT_DECAY)
    batches = [O.synthetic_rays(n_rays, seed=100 + i) for i in range(2)]

    def step(i):
        ro, rd, tgt = batches[i % len(batches)]
        target = tgt[:, :3] * tgt[:, 3:4] + bg * (1.0 - tgt[:, 3:4])
        loss = torch.nn.functional.mse_loss(render(ro, rd), target)
        loss = loss + torch.mean(torch.abs(table[1:] - table[:-1])) * TV_WEIGHT
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_([table], 1.0)
        torch.nn.utils.clip_grad_norm_([p for p in params if p is not table], 1.0)
        opt.step()
        return float(loss.detach())

    for i in range(warmup):
        step(i)
    times = []
    for i in range(steps):
        t0 = time.perf_counter()
        step(i)
        times.append(time.perf_counter() - t0)
    dt = sorted(times)[len(times) // 2]                     # median step (BASELINE.md section 2)
    return dict(value=n_rays / dt, unit="rays/s", cores=torch.get_num_threads(), kind=kind,
                sample=f"median of {steps} training steps of {n_rays} rays x {N_SAMPLES} samples ({occupancy} occupancy; "
                       f"the GPU arm runs 2^18 rays per step: reduced for memory and time), "
                       f"{'reference src/ + tcnn shim' if kind == 'reference' else 'oracle port'}, torch CPU fp32, "
                       f"after {warmup} warm-up", ms_per_step=1e3 * dt)


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    steps, warm = args.steps, args.warmup
    r = cpu_train_rays_per_s(args.cpu_rays, steps, warm, args.occupancy)
    line = {
        "impl": "reference", "metric": "train_rays_per_s", "value": r["value"], "unit": "rays/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.cpu_rays),
        "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": r["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- helpers
DUMP_MAX_ELEMENTS = 2 ** 20        # per array: C2 dumps 10 arrays, so a dump is at most 40 MB


def dump_outputs(out_dir, arrays):
    """``arrays`` (name -> tensor) as out_dir/<name>.npy in float32.  A tensor of more than DUMP_MAX_ELEMENTS elements is
    flattened and sampled at the same seeded positions in every run."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_ELEMENTS].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def workload_config(args, rays):
    return {
        "workload": "C2 Part-2 Instant-NeRF training step: hash grid L=16 F=2 T=2^19 + 64-wide sigma/color MLPs "
                    "+ 128^3 occupancy grid, synthetic 800x800 NeRF-Synthetic-shaped rays, AdamW + TV loss",
        "rays_per_gpu": rays, "n_samples": N_SAMPLES, "occupancy": args.occupancy,
        "occupancy_note": "dense = all voxels active (the reference's warm-up state, 100 % of samples evaluated); "
                          "sparse = ball r=0.75 (~6.5 % of voxels)",
        "l2": "per-step working set (activations, GBs) far exceeds the 126 MB L2; no explicit flush; "
              "a fresh jitter draw and a rotating ray batch every step",
        "parallelism": f"dp{args.gpus} (rays sharded, weights+tables replicated, one gradient all-reduce per step)",
    }


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(index)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.03 <= t <= t1 + 0.03] or [r for t, r in self.rows if t >= t0 - 1.0]
        sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in rows)]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(rows[0][1]) if rows and rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max(pw) if pw else None, "samples": len(rows), "reasons": reasons}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


def ncu_units(kernel_name):
    """per-unit utilisation (DRAM / L2 / L1TEX / tensor pipe, % of peak) of the dominant entry point's kernels from the
    committed `ncu --set full` capture: which unit actually binds it."""
    p = os.path.join(ROOT, "profiles", "ncu_units.json")
    if os.path.exists(p):
        return json.load(open(p)).get(kernel_name)
    return None


def ncu_traffic(kernel_name):
    """dram bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if os.path.exists(p):
        return json.load(open(p)).get(kernel_name)
    return None


def _maybe_profile(step):
    """development aid (B2N_PROF=1 | cpu): per-kernel device time / per-op host time of 3 steps, to stderr"""
    if not os.environ.get("B2N_PROF"):
        return
    from torch.profiler import ProfilerActivity, profile
    cpu = os.environ["B2N_PROF"] == "cpu"
    with profile(activities=[ProfilerActivity.CUDA] + ([ProfilerActivity.CPU] if cpu else [])) as prof:
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
    print(prof.key_averages().table(sort_by="self_cpu_time_total" if cpu else "cuda_time_total", row_limit=40,
                                    max_name_column_width=70), file=sys.stderr)


def bench_c1(dev, steps):
    """BASELINE.json configs[0] ("C1", Part 2 vanilla NeRF: PosEnc 10/4, 8x256 MLP on tcgen05, 64 samples, batch
    4096) on one GPU -- reported as an extra, the headline stays C2."""
    from b2n import synthetic
    from src.core import NeuralField
    from src.renderer import render_rays
    torch.manual_seed(0)
    import b2n
    model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).to(dev).train()
    # run.py:305 trains Part 2 with torch.optim.Adam(lr=5e-4): AdamW with weight_decay = 0 is the same update, done here
    # by the package's two-launch fused optimizer (SURVEY 8f-2) instead of torch's multi-tensor kernels
    opt = b2n.optim.FusedAdamW(model.parameters(), lr=5e-4, weight_decay=0.0)
    B, N = 4096, 64
    pool = [tuple(t.to(dev) for t in synthetic.random_rays(B, seed=50 + i)) for i in range(3)]

    def step(i):
        ro, rd, tgt = pool[i % 3]
        target = tgt[:, :3] * tgt[:, 3:4] + (1.0 - tgt[:, 3:4])
        pred, _, _ = render_rays(model, ro, rd, NEAR, FAR, N, True, white_bkgd=True)
        loss = torch.nn.functional.mse_loss(pred, target)
        opt.zero_grad()
        loss.backward()
        opt.step()

    def run(fn, n, warm):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    ms_train = run(step, steps, 5)
    _maybe_profile(step)
    # the same step captured into ONE CUDA graph (b2n.graphs): no occupancy grid -> every shape is static.  A fresh model
    # and a capturable Adam; per step the new ray batch is copied into the graph's static input buffers.
    graph = {}
    try:
        import b2n
        torch.manual_seed(0)
        gmodel = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).to(dev).train()
        gopt = b2n.optim.FusedAdamW(gmodel.parameters(), lr=5e-4, weight_decay=0.0)

        def gstep(ro, rd, tgt):
            target = tgt[:, :3] * tgt[:, 3:4] + (1.0 - tgt[:, 3:4])
            pred, _, _ = render_rays(gmodel, ro, rd, NEAR, FAR, N, True, white_bkgd=True)
            loss = torch.nn.functional.mse_loss(pred, target)
            gopt.zero_grad(set_to_none=True)
            loss.backward()
            gopt.step()
            return loss

        graphed = b2n.graphs.GraphedStep(gstep, pool[0])
        ms_graph = run(lambda i: graphed(*pool[i % 3]), steps, 5)
        graph = {"train_rays_per_s_cuda_graph": B / ms_graph * 1e3, "train_ms_per_step_cuda_graph": ms_graph,
                 "cuda_graph_note": "whole step (march .. fused Adam) replayed as one graph launch",
                 "loss_after_graph_steps": float(graphed(*pool[0]).detach())}
    except Exception as exc:        # reported, never hidden: the eager numbers above stand on their own
        graph = {"cuda_graph_error": f"{type(exc).__name__}: {exc}"[:300]}
    model.eval()
    with torch.no_grad():
        ms_render = run(lambda i: render_rays(model, pool[i % 3][0], pool[i % 3][1], NEAR, FAR, N, False), steps, 5)
    return {"workload": "C1 Part-2 vanilla NeRF, B=4096 rays x 64 samples, 8x256 MLP (tcgen05 bf16), Adam (b2n.optim.FusedAdamW, weight_decay 0)",
            "train_rays_per_s": B / ms_train * 1e3, "train_ms_per_step": ms_train,
            "train_mlp_tflops_algorithmic": 3 * 2.0 * B * N * 593408 / ms_train / 1e9,
            "render_msamples_per_s": B * N / ms_render * 1e3 / 1e6, **graph}


DYNAMIC = {
    # BASELINE.json configs[2..4]; shapes from configs/part3.yaml.example, part3_instant.yaml.example, part4.yaml.example
    "c3_dnerf": dict(cfg=dict(mode="part3", L_embed_time=10, L_embed=10, deform_hidden_dim=128, deform_num_layers=4,
                              canonical_type="nerf", L_embed_canon=10, hidden_dim=256, num_layers=8, skip_layer=4,
                              view_dim=128), B=2048, N=64, grid=None, lr=5e-4, reg=1e-4, tv=0.0,
                     label="C3 Part-3 standard D-NeRF (Fourier-MLP deformation 4x128 + Fourier-MLP canonical 8x256)"),
    "c4_instant_dnerf": dict(cfg=dict(mode="part3", L_embed_time=10, L_embed=10, deform_hidden_dim=128,
                                      deform_num_layers=4, canonical_type="instant", n_levels=16,
                                      n_features_per_level=2, log2_hashmap_size=19, base_resolution=16,
                                      per_level_scale=1.5, scene_bound=1.5, hidden_dim=64, use_coord_noise=True,
                                      coord_noise_std=0.005, time_noise_std=0.04),
                             B=8192, N=128, grid=(128, 0.01), lr=5e-3, reg=1e-2, tv=1e-5,
                             label="C4 Part-3 Instant D-NeRF (Fourier-MLP deformation + hash-grid canonical, 128^3 grid)"),
    "c5_dualhash": dict(cfg=dict(mode="part4", deform_n_levels=12, deform_n_features_per_level=2,
                                 deform_log2_hashmap_size=16, deform_base_resolution=16, deform_per_level_scale=1.5,
                                 deform_hidden_dim=64, L_embed_time=10, time_modulation_dim=64,
                                 time_modulation_layers=2, n_levels=16, n_features_per_level=2, log2_hashmap_size=20,
                                 base_resolution=16, per_level_scale=1.5, scene_bound=1.5, hidden_dim=64,
                                 use_coord_noise=True, coord_noise_std=0.001, time_noise_std=0.01),
                        B=8192, N=64, grid=(64, 0.01), lr=1e-2, reg=1e-4, tv=1e-6,
                        label="C5 Part-4 Dual-Hash dynamic NeRF (3 deformation hash grids + time modulation + canonical hash grid)"),
}


def bench_dynamic(dev, name, steps, warm=4, occupancy="dense", world=1, rank=0, strong=False):
    """Training step of run.py:1073-1178 / :1804-1949 (autocast + GradScaler, render_rays with times, RGB MSE +
    deformation L2 + table TV, clip, AdamW) for the dynamic configs -- reported as extras.

    world > 1: ray-sharded data parallel (replicated weights / tables, one flat gradient buffer averaged over ranks
    before unscale / clip / AdamW; every rank must call this).  ``strong``: the config's batch is the GLOBAL batch
    (B / world rays per GPU, BASELINE.json configs[4]: 8192 rays sharded over the GPUs); otherwise B rays per GPU (weak).

    Legs: torch AdamW (the reference's optimizer calls, world == 1 only), b2n.optim.FusedAdamW (TV + unscale + clip +
    AdamW as two launches; any world), and on one GPU the whole step as ONE CUDA graph (static-capacity march: no host
    read of the active-sample count, b2n.march.set_static_capacity)."""
    import torch.distributed as dist
    import b2n
    from b2n import march, synthetic
    from b2n.dp import GradAllReducer
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays
    spec = DYNAMIC[name]
    torch.manual_seed(0)
    model = NeuralField(spec["cfg"]).to(dev).train()
    B, N = spec["B"], spec["N"]
    if strong:
        B = B // world
    grid = None
    if spec["grid"]:
        grid = DensityGrid(resolution=spec["grid"][0], bound=1.5, threshold=spec["grid"][1]).to(dev)
        if occupancy == "sparse":
            grid.binary_grid = synthetic.ball_occupancy(spec["grid"][0], 1.5).to(dev)
    reducer = GradAllReducer(model, world, direct=True) if world > 1 else None      # no TV term in the loss below: FusedAdamW carries it
    pool = [tuple(t.to(dev) for t in synthetic.random_rays(B, seed=70 + i + 1000 * rank, n_views=150, with_time=True))
            for i in range(3)]
    bg = torch.ones(3, device=dev)
    tables = [m.encoding.params for n_, m in model.named_children() if hasattr(m, "encoding") and n_ != "deformation_grid"]
    table_ids = {id(t) for t in tables}

    def loss_of(batch, with_tv):
        ro, rd, tgt, times = batch
        target = tgt[:, :3] * tgt[:, 3:4] + bg * (1.0 - tgt[:, 3:4])
        with torch.amp.autocast("cuda", enabled=True):
            pred, _, _, extras = render_rays(model=model, rays_o=ro, rays_d=rd, near=NEAR, far=FAR, n_samples=N,
                                             perturb=True, times=times, density_grid=grid, bg_color=bg)
            loss = torch.nn.functional.mse_loss(pred, target) + torch.mean(extras["mean_delta_x"] ** 2) * spec["reg"]
            if with_tv and spec["tv"] > 0:
                for tb in tables:
                    loss = loss + torch.mean(torch.abs(tb[1:] - tb[:-1])) * spec["tv"]
        return loss

    def sync():
        if world > 1:
            dist.barrier(device_ids=[dev.index])
        torch.cuda.synchronize()

    def run(fn, n, w):
        for i in range(w):
            fn(i)
        sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        sync()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / n

    out = {"workload": f"{spec['label']}, B={B} rays x {N} samples per GPU"
                       f"{' (= %d global, strong scaling)' % (B * world) if strong else ''}, AMP autocast + GradScaler, "
                       f"AdamW, {occupancy} occupancy", "n_gpus": world}
    # ---- (1) the reference's optimizer calls: torch AdamW + unscale_ + clip_grad_norm_ + TV term in the loss
    if world == 1:
        opt = torch.optim.AdamW(model.parameters(), lr=spec["lr"], weight_decay=1e-5)
        scaler = torch.amp.GradScaler("cuda", enabled=True)

        def step(i):
            loss = loss_of(pool[i % 3], True)
            opt.zero_grad()
            scaler.scale(loss).backward()
            scaler.unscale_(opt)
            torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=1.0)
            scaler.step(opt)
            scaler.update()

        ms_train = run(step, steps, warm)
        _maybe_profile(step)
        out.update(train_rays_per_s=B / ms_train * 1e3, train_ms_per_step=ms_train)
    # ---- (2) b2n.optim.FusedAdamW (SURVEY 8f-2): the loss carries no TV term, scaler.step() hands the loss scale / inf
    # flag to the optimizer; under data parallelism the gradients are averaged first, so every rank takes the same
    # inf / clip decisions
    fopt = b2n.optim.FusedAdamW(
        [{"params": [p for p in model.parameters() if id(p) in table_ids], "tv_weight": spec["tv"]},
         {"params": [p for p in model.parameters() if id(p) not in table_ids]}], lr=spec["lr"], weight_decay=1e-5)
    fscaler = torch.amp.GradScaler("cuda", enabled=True)

    def fstep(i):
        loss = loss_of(pool[i % 3], False)
        if reducer is None:
            fopt.zero_grad()
        else:
            reducer.zero_grad()
        fscaler.scale(loss).backward()
        if reducer is not None:
            reducer.allreduce()
        fscaler.step(fopt, max_norm=1.0)
        fscaler.update()

    try:
        ms_fused = run(fstep, steps, warm)
        out.update(train_rays_per_s_fused_optimizer=world * B / ms_fused * 1e3, train_ms_per_step_fused_optimizer=ms_fused)
        if world > 1:
            out.update(train_rays_per_s=world * B / ms_fused * 1e3, train_ms_per_step=ms_fused)
    except Exception as exc:
        out["fused_optimizer_error"] = f"{type(exc).__name__}: {exc}"[:300]
    if reducer is not None:
        # the collective on its own: the flat gradient buffer all-reduced back to back (what a step pays when nothing overlaps)
        ms_ar = run(lambda i: reducer.allreduce(), steps, 3)
        out.update(allreduce_bytes_per_step=reducer.nbytes, allreduce_ms_alone=ms_ar)
    # ---- (3) the whole step as ONE CUDA graph (static-capacity march + FusedAdamW; constant LR inside the graph).  Under
    # data parallelism the gradient all-reduces (NCCL) are captured with it: at 1024 rays per GPU (C5 strong scaling at 8
    # GPUs) the eager step is launch-bound, the replay is not
    if world == 1 or os.environ.get("B2N_DP_GRAPH", "1") == "1":
        try:
            march.set_static_capacity(True)
            gopt = b2n.optim.FusedAdamW(
                [{"params": [p for p in model.parameters() if id(p) in table_ids], "tv_weight": spec["tv"]},
                 {"params": [p for p in model.parameters() if id(p) not in table_ids]}], lr=spec["lr"], weight_decay=1e-5)
            gscaler = torch.amp.GradScaler("cuda", enabled=True)
            if reducer is None:
                for p in model.parameters():
                    p.grad = torch.zeros_like(p)

            def gstep(ro, rd, tgt, times):
                loss = loss_of((ro, rd, tgt, times), False)
                if reducer is None:
                    for p in model.parameters():
                        p.grad.zero_()
                else:
                    reducer.zero_grad()
                gscaler.scale(loss).backward()
                if reducer is not None:
                    reducer.allreduce()
                gscaler.step(gopt, max_norm=1.0)
                gscaler.update()
                return loss

            ms_static = run(lambda i: gstep(*pool[i % 3]), steps, warm)          # static capacity, eager launches
            graphed = b2n.graphs.GraphedStep(gstep, pool[0])
            ms_graph = run(lambda i: graphed(*pool[i % 3]), steps, warm)
            b2n.check_errors()
            out.update(train_rays_per_s_static_capacity=world * B / ms_static * 1e3,
                       train_rays_per_s_cuda_graph=world * B / ms_graph * 1e3,
                       train_ms_per_step_cuda_graph=ms_graph, loss_after_graph_steps=float(graphed(*pool[0]).detach()))
        except Exception as exc:
            out["cuda_graph_error"] = f"{type(exc).__name__}: {exc}"[:300]
        finally:
            march.set_static_capacity(False)
            if reducer is None:
                for p in model.parameters():
                    p.grad = None
    model.eval()
    with torch.no_grad():
        ms_render = run(lambda i: render_rays(model, pool[i % 3][0], pool[i % 3][1], NEAR, FAR, N, False,
                                              times=pool[i % 3][3], density_grid=grid, bg_color=bg), steps, 2)
    out["render_msamples_per_s"] = world * B * N / ms_render * 1e3 / 1e6
    if reducer is not None:
        reducer.remove_hooks()
    return out


# --------------------------------------------------------------------------------------- GPU arm
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)

    import torch.distributed as dist
    import b2n
    from b2n import _lib, synthetic
    from b2n.dp import GradAllReducer
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_rays

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b2n) needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "NONE"       # keep stdout to the single JSON line (no "NCCL version" banner)
        dist.init_process_group("nccl", device_id=dev)
    B = args.rays
    if args.only:
        r = (bench_c1(dev, args.steps) if args.only == "c1_vanilla"
             else bench_dynamic(dev, args.only, args.steps, occupancy=args.occupancy))
        print(json.dumps({args.only: r}), flush=True)
        return

    torch.manual_seed(0)                                   # replicated init on every rank
    model = NeuralField(C2).to(dev).train()
    table = model.representation.encoding.params

    def make_grid(kind):
        g = DensityGrid(resolution=GRID_R, bound=1.5, threshold=GRID_THR).to(dev)
        if kind == "sparse":
            g.binary_grid = synthetic.ball_occupancy(GRID_R, 1.5).to(dev)
        return g

    opt = torch.optim.AdamW(model.parameters(), lr=LR, weight_decay=WEIGHT_DECAY)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=TRAIN_ITERS, eta_min=ETA_MIN)
    # flat gradient buffer: one memset, all-reduce of element ranges as they become final.  The headline step keeps the
    # reference's TV term in the loss (an autograd-side gradient on the table), so its table is reduced from the
    # post-accumulate hook; the fused-optimizer leg (TV inside FusedAdamW) uses the direct sinks
    reducer = GradAllReducer(model, world)
    bg = torch.ones(3, device=dev)

    n_pool = 3
    host_pool = [tuple(t.pin_memory() for t in synthetic.random_rays(B, seed=1000 * rank + i)) for i in range(n_pool)]
    dev_pool = [tuple(t.to(dev) for t in b) for b in host_pool]
    h2d_bytes = sum(t.numel() * t.element_size() for t in host_pool[0])

    last = {}                                              # what the latest train_step computed (--dump-outputs)

    def train_step(batch, grid):
        rays_o, rays_d, rgba = batch
        target = rgba[:, :3] * rgba[:, 3:4] + bg * (1.0 - rgba[:, 3:4])
        pred, depth, acc = render_rays(model=model, rays_o=rays_o, rays_d=rays_d, near=NEAR, far=FAR,
                                       n_samples=N_SAMPLES, perturb=True, white_bkgd=True, density_grid=grid, bg_color=bg)
        loss_rgb = torch.nn.functional.mse_loss(pred, target)
        loss = loss_rgb + torch.mean(torch.abs(table[1:] - table[:-1])) * TV_WEIGHT
        reducer.zero_grad()
        loss.backward()
        reducer.allreduce()
        torch.nn.utils.clip_grad_norm_(model.representation.parameters(), max_norm=1.0)
        torch.nn.utils.clip_grad_norm_(model.decoder.parameters(), max_norm=1.0)
        opt.step()
        sched.step()
        last.update(color=pred.detach(), depth=depth.detach(), acc=acc.detach(), loss=loss.detach())
        return loss

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local])
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    # ---- headline: device-resident batches, profiler + clock sampler on
    grid = make_grid(args.occupancy)
    sampler = ClockSampler(local) if rank == 0 else None      # started early: nvidia-smi needs ~1 s to start
    for i in range(args.warmup):
        train_step(dev_pool[i % n_pool], grid)
    barrier()
    prof = _lib.Profiler()
    _lib.PROFILER = prof
    launches0 = _lib.LAUNCHES["count"]
    t_wall0 = time.time()
    ms = timed(lambda i: train_step(dev_pool[i % n_pool], grid), args.steps, 0)
    t_wall1 = time.time()
    _lib.PROFILER = None
    launches = _lib.LAUNCHES["count"] - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    value = world * B * args.steps / (ms * 1e-3)
    summary = prof.summary()
    if args.dump_outputs and rank == 0:
        params = list(model.named_parameters())
        dump_outputs(args.dump_outputs, {**last, **{f"param.{n}": p for n, p in params},
                                         **{f"grad.{n}": p.grad for n, p in params}})

    # ---- e2e: pinned host batch -> H2D -> step -> D2H loss, every step
    def e2e_step(i):
        hb = host_pool[i % n_pool]
        batch = tuple(t.to(dev, non_blocking=True) for t in hb)
        return float(train_step(batch, grid).item())

    ms_e2e = timed(e2e_step, args.steps, 1)
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)

    extras = {}
    if not args.no_extras:
        # ---- the other occupancy case
        other = "sparse" if args.occupancy == "dense" else "dense"
        g2 = make_grid(other)
        ms2 = timed(lambda i: train_step(dev_pool[i % n_pool], g2), args.steps, 2)
        extras[f"train_rays_per_s_{other}"] = world * B * args.steps / (ms2 * 1e-3)
        # ---- the same step with the TV term, the two per-group clips and AdamW inside b2n.optim.FusedAdamW (SURVEY 8f-2)
        try:
            import b2n
            fopt = b2n.optim.FusedAdamW(
                [{"params": list(model.representation.parameters()), "tv_weight": TV_WEIGHT, "max_norm": 1.0},
                 {"params": list(model.decoder.parameters()), "max_norm": 1.0}], lr=LR, weight_decay=WEIGHT_DECAY)

            if world > 1:
                reducer.remove_hooks()
                reducer = GradAllReducer(model, world, direct=True)     # table gradient written in place, fine levels reduced early

            def fused_step(batch):
                rays_o, rays_d, rgba = batch
                target = rgba[:, :3] * rgba[:, 3:4] + bg * (1.0 - rgba[:, 3:4])
                pred, _, _ = render_rays(model=model, rays_o=rays_o, rays_d=rays_d, near=NEAR, far=FAR,
                                         n_samples=N_SAMPLES, perturb=True, white_bkgd=True, density_grid=grid, bg_color=bg)
                loss = torch.nn.functional.mse_loss(pred, target)
                reducer.zero_grad()
                loss.backward()
                reducer.allreduce()
                fopt.step()

            ms4 = timed(lambda i: fused_step(dev_pool[i % n_pool]), args.steps, 2)
            extras["train_rays_per_s_fused_optimizer"] = world * B * args.steps / (ms4 * 1e-3)
        except Exception as exc:
            extras["fused_optimizer_error"] = f"{type(exc).__name__}: {exc}"[:300]
        # ---- one GPU: the C2 step with NO host read of the active-sample count (static-capacity march), eager and as ONE
        # CUDA graph (constant LR inside the graph)
        if world == 1:
            from b2n import march as _march
            try:
                _march.set_static_capacity(True)
                for p in model.parameters():
                    p.grad = torch.zeros_like(p)
                gopt = b2n.optim.FusedAdamW(
                    [{"params": list(model.representation.parameters()), "tv_weight": TV_WEIGHT, "max_norm": 1.0},
                     {"params": list(model.decoder.parameters()), "max_norm": 1.0}], lr=LR, weight_decay=WEIGHT_DECAY)

                def gstep(rays_o, rays_d, rgba):
                    target = rgba[:, :3] * rgba[:, 3:4] + bg * (1.0 - rgba[:, 3:4])
                    pred, _, _ = render_rays(model=model, rays_o=rays_o, rays_d=rays_d, near=NEAR, far=FAR,
                                             n_samples=N_SAMPLES, perturb=True, white_bkgd=True, density_grid=grid, bg_color=bg)
                    loss = torch.nn.functional.mse_loss(pred, target)
                    for p in model.parameters():
                        p.grad.zero_()
                    loss.backward()
                    gopt.step()
                    return loss

                ms5 = timed(lambda i: gstep(*dev_pool[i % n_pool]), args.steps, 2)
                extras["train_rays_per_s_static_capacity"] = B * args.steps / (ms5 * 1e-3)
                graphed = b2n.graphs.GraphedStep(gstep, dev_pool[0])
                ms6 = timed(lambda i: graphed(*dev_pool[i % n_pool]), args.steps, 2)
                extras["train_rays_per_s_cuda_graph"] = B * args.steps / (ms6 * 1e-3)
                extras["loss_after_graph_steps"] = float(graphed(*dev_pool[0]).detach())
                del graphed
            except Exception as exc:
                extras["cuda_graph_error"] = f"{type(exc).__name__}: {exc}"[:300]
            finally:
                _march.set_static_capacity(False)
                reducer_views = reducer._views
                for p in model.parameters():
                    p.grad = reducer_views[p].view_as(p)
        # ---- render Msamples/s (forward only, no jitter, no_grad)
        model.eval()
        with torch.no_grad():
            def render(i):
                ro, rd, _ = dev_pool[i % n_pool]
                render_rays(model, ro, rd, NEAR, FAR, N_SAMPLES, False, density_grid=grid, bg_color=bg)
            ms3 = timed(render, args.steps, 2)
        model.train()
        extras["render_msamples_per_s"] = world * B * N_SAMPLES * args.steps / (ms3 * 1e-3) / 1e6
        extras["render_occupancy"] = args.occupancy

    if not args.no_extras and rank == 0:
        # L2 random-gather peak measured live (SURVEY 8d: MEASURED_PEAKS.json has no L2 figure; the hash-grid kernels are
        # gathers / reductions over a table that lives in L2, so this is the peak they are to be read against)
        from b2n._lib import call as _call, ptr as _ptr, stream as _stream
        sink = torch.zeros(1, device=dev)
        l2 = {}
        for mib, log2n in ((32, 22), (64, 23)):
            tab = torch.randn(1 << log2n, 2, device=dev)
            blocks, per_thread = 148 * 16, 512
            best = 1e9
            for i in range(4):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _call("b2n_debug_gather_bench", _ptr(tab), 1 << log2n, blocks, per_thread, _ptr(sink), _stream())
                e1.record()
                torch.cuda.synchronize()
                if i:
                    best = min(best, e0.elapsed_time(e1))
            l2[f"table_{mib}MiB_Ggathers_per_s"] = blocks * 256 * per_thread / best / 1e6
            del tab
        n_active = summary.get("b2n_hash_fwd", {}).get("bytes", 0.0) / args.steps / (12 + 16 * 2 * 4 * 9)   # points per step
        per_step = {k: summary[k]["ms"] / args.steps for k in ("b2n_hash_fwd", "b2n_hash_bwd") if k in summary}
        extras["hash_vs_l2"] = {
            "l2_random_8B_gather_peak": l2,
            "active_points_per_step": n_active,
            "hash_fwd_corner_gathers_Gps": n_active * 16 * 8 / per_step.get("b2n_hash_fwd", float("inf")) / 1e6,
            "hash_bwd_corner_reductions_Gps": n_active * 16 * 8 / per_step.get("b2n_hash_bwd", float("inf")) / 1e6,
            "note": "8 corners x 16 levels per point; x-neighbour corner pairs that are adjacent table entries move as ONE "
                    "16-byte access, and the coarse levels hit in L1, so the corner rate can exceed the 8-byte gather peak"}
    dp_scalars = {}
    if not args.no_extras and world > 1:
        # BASELINE.json configs[4]: Part 4 Dual-Hash, ray batch sharded over the GPUs, hash-table gradient all-reduce:
        # weak scaling (8192 rays per GPU) and the config's own global batch of 8192 rays split over the GPUs (strong)
        weak = bench_dynamic(dev, "c5_dualhash", args.steps, world=world, rank=rank)
        strong = bench_dynamic(dev, "c5_dualhash", args.steps, world=world, rank=rank, strong=True)
        extras["c5_dualhash_dp"] = weak
        extras["c5_dualhash_dp_strong"] = strong
        dp_scalars = {"c5_dualhash_dp_weak_rays_per_s": weak.get("train_rays_per_s"),
                      "c5_dualhash_dp_weak_ms_per_step": weak.get("train_ms_per_step"),
                      "c5_dualhash_dp_strong_rays_per_s": strong.get("train_rays_per_s"),
                      "c5_dualhash_dp_strong_ms_per_step": strong.get("train_ms_per_step"),
                      "c5_dualhash_dp_strong_cuda_graph_rays_per_s": strong.get("train_rays_per_s_cuda_graph"),
                      "c5_dualhash_dp_weak_cuda_graph_rays_per_s": weak.get("train_rays_per_s_cuda_graph"),
                      "c5_dualhash_dp_allreduce_ms_alone": weak.get("allreduce_ms_alone"),
                      "c5_dualhash_dp_allreduce_bytes": weak.get("allreduce_bytes_per_step")}
    if not args.no_extras and rank == 0:
        extras["c1_vanilla"] = bench_c1(dev, args.steps)
        for name in DYNAMIC:
            extras[name] = bench_dynamic(dev, name, args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, tensor_peak, peak_src = measured_peaks()
    kernels = sorted(({"entry": k, "calls_per_step": v["calls"] / args.steps, "ms_per_step": v["ms"] / args.steps,
                       "alg_gb_per_step": v["bytes"] / args.steps / 1e9,
                       "gbs": (v["bytes"] / 1e9) / (v["ms"] * 1e-3) if v["ms"] > 0 else None,
                       "tflops": (v["flops"] / 1e12) / (v["ms"] * 1e-3) if v["ms"] > 0 else None}
                      for k, v in summary.items()), key=lambda d: -d["ms_per_step"])
    # ---- rooflines.  Which unit bounds an entry point (DESIGN.md section 3):
    #   tensor : the fused 16-bit MLP kernels -- algorithmic FLOPs (unpadded MACs of SURVEY 8d, forward x3 for a training
    #            step) / time against the measured sustained 16-bit dense rate
    #   l2     : the hash-grid kernels -- the tables and the 52 MB gradient table live in L2; what is counted is 32-byte
    #            L2 SECTOR operations: 4 per (point, level) is the floor (8 corners = 4 x-neighbour pairs, each pair inside
    #            one sector at best), against the L2 random sector rate measured live below (gathers for the forward,
    #            red.global for the table gradient).  hbm_compulsory_frac = the bytes that must cross HBM (positions +
    #            feature / gradient rows) / time / HBM peak; alg_gbs = the SURVEY 8d byte figure / time
    #   hbm    : compositing, march, everything streaming
    from b2n._lib import call as _call, ptr as _ptr, stream as _stream
    l2_peaks = {}

    def l2_peak(kind):
        if kind in l2_peaks:
            return l2_peaks[kind]
        tab = torch.zeros(1 << 22, 2, device=dev)                  # 32 MiB float2 table: L2-resident
        sink = torch.zeros(1, device=dev)
        blocks, per_thread, best = 148 * 16, 256, 1e9
        for i in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            if kind == "gather":
                _call("b2n_debug_gather_bench", _ptr(tab), 1 << 22, blocks, per_thread, _ptr(sink), _stream())
            else:
                _call("b2n_debug_red_bench", _ptr(tab), 1 << 22, blocks, per_thread, 0, _stream())
            e1.record()
            torch.cuda.synchronize()
            if i:
                best = min(best, e0.elapsed_time(e1))
        l2_peaks[kind] = blocks * 256 * per_thread / best / 1e6          # G sector operations / s (one sector per lane)
        return l2_peaks[kind]

    n_points = summary.get("b2n_hash_fwd", {}).get("bytes", 0.0) / args.steps / (12 + 16 * 2 * 4 * 9)   # active points / step
    L_levels = C2["n_levels"]

    def roofline_of(k):
        ms_k = k["ms_per_step"] / max(k["calls_per_step"], 1e-9)
        base = {"kernel": k["entry"], "avg_launch_ms": ms_k, "share_of_step": k["ms_per_step"] / (ms / args.steps),
                "traffic": ncu_traffic(k["entry"]), "ncu": ncu_units(k["entry"])}
        if k["entry"] in ("b2n_hash_fwd", "b2n_hash_bwd") and n_points > 0:
            kind = "gather" if k["entry"] == "b2n_hash_fwd" else "red"
            peak = l2_peak(kind)
            ach = n_points * L_levels * 4 / (k["ms_per_step"] * 1e-3) / 1e9
            return {**base, "bound": "l2", "achieved": ach, "peak": peak, "unit": "G L2 sector-ops/s", "frac": ach / peak,
                    "peak_source": f"measured live: random {'8-byte gathers' if kind == 'gather' else 'red.global.add.v2.f32'} "
                                   "over a 32 MiB table, one 32-byte sector per lane",
                    "sectors_per_point_level": 4,
                    "hbm_compulsory_frac": n_points * (12 + L_levels * 2 * 4) / (k["ms_per_step"] * 1e-3) / 1e9 / hbm_peak,
                    "alg_gbs": k["gbs"]}
        if k["entry"].startswith(("b2n_instant_mlp", "b2n_fmlp", "b2n_nerf_mlp")) and k["tflops"]:
            return {**base, "bound": "tensor", "achieved": k["tflops"], "peak": tensor_peak, "unit": "TFLOP/s",
                    "frac": k["tflops"] / tensor_peak, "peak_source": peak_src + " (cuBLAS bf16 sustained; fp16 runs at the same rate)",
                    "alg_gbs": k["gbs"]}
        return {**base, "bound": "hbm", "achieved": k["gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": (k["gbs"] / hbm_peak) if k["gbs"] else None, "peak_source": peak_src}

    rooflines = [roofline_of(k) for k in kernels[:8]]
    roofline = rooflines[0]

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cpu_train_rays_per_s(args.cpu_rays, args.steps, args.warmup, args.occupancy)   # --cpu-rays bounds its cost
        cpu = {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")}

    line = {
        "metric": "train_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": workload_config(args, B),
        "clocks": clocks, "gpu_launches": launches,
        "e2e": {"value": e2e_value, "unit": "rays/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        **dp_scalars,
        "roofline": roofline, "rooflines": rooflines, "cpu_baseline": cpu, "kernels": kernels[:12],
    }
    line.update(extras)
    line.update({k + "_": v for k, v in dp_scalars.items()})      # repeated at the very end of the line (log tails)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
