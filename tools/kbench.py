#!/usr/bin/env python
"""Micro-timings of single entry points (CUDA events, L2-cold inputs) -- development aid.
    python tools/kbench.py mlp256 [P]
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "project-nerf_b200")]
import torch  # noqa: E402

import b2n  # noqa: E402
from b2n import _lib, ops  # noqa: E402
from src.core import NeuralField  # noqa: E402


def timeit(fn, n=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def mlp256(P):
    torch.manual_seed(0)
    model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().eval()
    xe = torch.randn(P, 63, device="cuda")
    de = torch.randn(P, 27, device="cuda")
    flops = 2.0 * P * 593408
    for pair in (0, 1):
        b2n._lib.lib.b2n_debug_mlp256_set_pair(pair)
        for save in (False, True):
            med, best = timeit(lambda: ops.nerf_mlp_forward(model.decoder, xe, de, save=save))
            print(f"mlp256 fwd pair={pair} P={P} save={save}: median {med:.3f} ms best {best:.3f} ms -> "
                  f"{flops / best / 1e9:.1f} TFLOP/s ({100 * flops / best / 1e9 / 1391.5:.1f} % of sustained bf16 peak)")
        _, _, _, err = ops.nerf_mlp_forward(model.decoder, xe, de, save=True)
        print(f"  err flag {int(err.item())}")
        # backward chain alone (data gradients): time the autograd call, minus nothing -- report the profiler's entry
        x2 = xe[: P].clone().requires_grad_(True)
        model.train()
        for it in range(6):
            if it == 1:
                b2n._lib.PROFILER = prof = b2n._lib.Profiler()
            r, s_ = model.decoder(x2, de)
            (r.sum() + s_.sum()).backward()
        torch.cuda.synchronize()
        b2n._lib.PROFILER = None
        for name, d in prof.summary().items():
            if "nerf_mlp" in name:
                print(f"    {name}: {d['ms'] / d['calls']:.3f} ms/call")
        model.eval()
    for pair in (0, 1):
        b2n._lib.lib.b2n_debug_mlp256_set_pair(pair)
        for what in ("fwd", "fwd+save", "bwd"):
            prof = torch.zeros(8 + 448, dtype=torch.int64, device="cuda")
            if what == "bwd":
                model.train()
                x2 = xe.clone().requires_grad_(True)
                r, s_ = model.decoder(x2, de)
                torch.cuda.synchronize()
                b2n._lib.lib.b2n_debug_mlp256_flags(16)
                b2n._lib.lib.b2n_debug_mlp256_prof(prof.data_ptr())
                (r.sum() + s_.sum()).backward()
                model.eval()
            else:
                b2n._lib.lib.b2n_debug_mlp256_flags(16)
                b2n._lib.lib.b2n_debug_mlp256_prof(prof.data_ptr())
                ops.nerf_mlp_forward(model.decoder, xe, de, save=what != "fwd")
            torch.cuda.synchronize()
            b2n._lib.lib.b2n_debug_mlp256_prof(None)
            b2n._lib.lib.b2n_debug_mlp256_flags(0)
            pr = prof.tolist()
            n = max(pr[4], 1)
            print(f"pair={pair} {what}: CTA0 cycles per tile pair ({pr[4]} pairs): whole {pr[7] / n:.0f} | pre-step {pr[5] / n:.0f}, "
                  f"bias staging {pr[6] / n:.0f}, epilogue-waits-MMA {pr[2] / n:.0f}, epilogue-body {pr[3] / n:.0f} | "
                  f"MMA-waits-epilogue {pr[0] / n:.0f}, MMA-waits-weights {pr[1] / n:.0f}")
    b2n._lib.lib.b2n_debug_mlp256_set_pair(1)
    with torch.no_grad():
        b2n.set_mlp_precision("fp32")
        med, best = timeit(lambda: model.decoder(xe, de), n=3, warm=1)
        print(f"fp32 layer-wise path: {best:.3f} ms -> {flops / best / 1e9:.1f} TFLOP/s")


def mlp256x(P):
    """role isolation of k_mlp256 (debug flags): kernel time of forward / backward with the epilogue drain and / or the MMAs removed"""
    torch.manual_seed(0)
    model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().train()
    xe = torch.randn(P, 63, device="cuda")
    de = torch.randn(P, 27, device="cuda")
    lib = b2n._lib.lib
    for pair in (0, 1):
        lib.b2n_debug_mlp256_set_pair(pair)
        for dbg in [int(v) for v in os.environ.get("KB_DBG", "0,1,2,3,7,15").split(",")]:
            lib.b2n_debug_mlp256_flags(dbg)
            x2 = xe.clone().requires_grad_(True)
            for it in range(5):
                if it == 1:
                    b2n._lib.PROFILER = prof = b2n._lib.Profiler()
                r, s_ = model.decoder(x2, de)
                (r.sum() + s_.sum()).backward()
                with torch.no_grad():
                    ops.nerf_mlp_forward(model.decoder, xe, de, save=False)
            torch.cuda.synchronize()
            b2n._lib.PROFILER = None
            lib.b2n_debug_mlp256_flags(0)
            ms = {}
            for name, nbytes, flops, e0, e1 in prof.records:
                if name in ("b2n_nerf_mlp_fwd", "b2n_nerf_mlp_bwd"):
                    key = name[-3:] + ("+save" if nbytes > P * 1000 and name.endswith("fwd") else "")
                    ms.setdefault(key, []).append(e0.elapsed_time(e1))
            print(f"pair={pair} dbg={dbg} ({ {0: 'full', 1: 'no drain', 2: 'no MMA', 3: 'handshakes + weight stream only', 7: 'handshakes only', 15: 'handshakes only, no row loads/stores'}[dbg]}): " +
                  ", ".join(f"{k} {min(v):.3f} ms" for k, v in sorted(ms.items())))
    lib.b2n_debug_mlp256_set_pair(1)


def mlp256t(P):
    """timeline of CTA 0's third tile pair (B2N_TRACE): per step / tile, cycles relative to the pair's first event"""
    torch.manual_seed(0)
    model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().train()
    xe = torch.randn(P, 63, device="cuda")
    de = torch.randn(P, 27, device="cuda")
    lib = b2n._lib.lib
    names = ["epi:wait", "epi:acc", "epi:done", "mma:wait", "mma:act", "mma:w0", "mma:issued", "epi:stage"]
    for pair, what, cta in ((0, "bwd", 0), (1, "fwd+save", 0), (1, "bwd", 0), (1, "bwd", 1)):
        lib.b2n_debug_mlp256_set_pair(pair)
        lib.b2n_debug_mlp256_flags(32 * cta)
        if True:
            x2 = xe.clone().requires_grad_(True)
            for _ in range(2):
                r, s_ = model.decoder(x2, de)
                (r.sum() + s_.sum()).backward()
            torch.cuda.synchronize()
            prof = torch.zeros(8 + 448, dtype=torch.int64, device="cuda")
            if what == "bwd":
                r, s_ = model.decoder(x2, de)
                torch.cuda.synchronize()
                lib.b2n_debug_mlp256_prof(prof.data_ptr())
                (r.sum() + s_.sum()).backward()
            else:
                lib.b2n_debug_mlp256_prof(prof.data_ptr())
                ops.nerf_mlp_forward(model.decoder, xe, de, save=True)
            torch.cuda.synchronize()
            lib.b2n_debug_mlp256_prof(None)
            tr = prof[8:].view(14, 2, 16)[:, :, :8].cpu()
            t00 = int(tr[tr > 0].min())
            print(f"--- pair={pair} {what} CTA {cta}: cycles since the first event of the pair; columns = {names}")
            for s in range(14):
                for t in range(2):
                    row = tr[s, t]
                    if int(row.max()) == 0:
                        continue
                    print(f"  step {s:2d} tile {t}: " + " ".join(f"{(int(v) - t00) if v > 0 else -1:7d}" for v in row))
    lib.b2n_debug_mlp256_set_pair(1)
    lib.b2n_debug_mlp256_flags(0)


def occ_update():
    """DensityGrid.update (SURVEY 8f-3): sigma-only sweep through NeuralField.density against the reference-style sweep
    through the full model (zero view directions, rgb dropped), C2 / C4 / C5 shapes, bf16 mode."""
    from src.renderer import DensityGrid

    class NoDensity(torch.nn.Module):
        def __init__(self, m):
            super().__init__()
            self.m, self.mode = m, m.mode

        def forward(self, *a, **k):
            return self.m(*a, **k)

    b2n.set_mlp_precision("bf16")
    cfgs = {
        "C2 part2_instant R=128": (dict(mode="part2_instant", scene_bound=1.5), 128, None),
        "C4 part3 instant R=128": (dict(mode="part3", canonical_type="instant", scene_bound=1.5), 128, 0.3),
        "C5 part4 R=64": (dict(mode="part4", scene_bound=1.5, log2_hashmap_size=20, deform_n_levels=12,
                               deform_log2_hashmap_size=16), 64, None),
    }
    for name, (cfg, R, tval) in cfgs.items():
        torch.manual_seed(0)
        model = NeuralField(cfg).cuda().eval()
        for label, mdl in (("density branch", model), ("full forward", NoDensity(model))):
            grid = DensityGrid(resolution=R, bound=1.5, threshold=0.01).cuda()
            t = None if tval is None else torch.tensor([[tval]], device="cuda")
            p0 = next(model.parameters())

            def once():
                with torch.no_grad():
                    p0.add_(0.0)                 # an optimizer step happened: version counter bumped, sweep cache invalid
                grid.update(mdl, device="cuda", time=t)

            def trio():                          # run.py:1972-1986: three update() calls in a row between two optimizer steps
                with torch.no_grad():
                    p0.add_(0.0)
                for _ in range(3):
                    grid.update(mdl, device="cuda", time=t, decay=0.95)
            med, best = timeit(once, n=5, warm=2)
            med3, best3 = timeit(trio, n=5, warm=2)
            print(f"occ update {name}: {label}: one call median {med:.3f} ms best {best:.3f} ms; "
                  f"three calls in a row (run.py pattern) median {med3:.3f} ms")


def mesh(sizes=(128, 256, 512)):
    """b2n.mesh: the sigma sweep of the C2 model (part2_instant, scene_bound 1.5, bf16 mode, density branch) on an R^3
    lattice, and surface extraction alone on an analytic field (a ball of radius 0.6 in [-1, 1]^3, sigma = 1 + 4 * signed
    distance, tau = 1; count / emit split from per-entry CUDA events).  Medians over 10 runs after 3 warm-ups."""
    import subprocess
    from b2n import mesh as bm
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                # noqa: BLE001 -- the measurement stands without it
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, power.max_limit: {smi}")
    b2n.set_mlp_precision("bf16")
    torch.manual_seed(0)
    model = NeuralField(dict(mode="part2_instant", scene_bound=1.5)).cuda().eval()
    for R in sizes:
        med, best = timeit(lambda: bm.density_lattice(model, R, 1.5), n=10, warm=3)
        print(f"sweep C2 part2_instant R={R}: {R ** 3 / 1e6:.1f} M points, median {med:.3f} ms (best {best:.3f}), "
              f"{R ** 3 / med / 1e6:.2f} G points/s")
    for R in sizes:
        ax = bm.lattice_axis(R, 1.0, "cuda").double()
        x, y, z = torch.meshgrid(ax, ax, ax, indexing="ij")
        sigma = (1.0 + 4.0 * (0.6 - torch.sqrt(x * x + y * y + z * z))).float().contiguous()
        del x, y, z
        verts, faces = bm.extract(sigma, 1.0, 1.0)
        med, best = timeit(lambda: bm.extract(sigma, 1.0, 1.0), n=10, warm=3)
        _lib.PROFILER = _lib.Profiler()
        for _ in range(10):
            bm.extract(sigma, 1.0, 1.0)
        torch.cuda.synchronize()
        summ = _lib.PROFILER.summary()
        _lib.PROFILER = None
        split = ", ".join(f"{k[len('b2n_mesh_'):]} {v['ms'] / v['calls']:.3f} ms" for k, v in summ.items())
        print(f"extract ball R={R}: {verts.shape[0]} vertices, {faces.shape[0]} triangles, median {med:.3f} ms "
              f"(best {best:.3f}; {split}; the rest is the host read of the totals and the allocations)")
        del sigma, verts, faces
        torch.cuda.empty_cache()


def render(H=800, N=128, chunk=2 ** 16, checkpoints=(300, 2000)):
    """One 800 x 800 view at N = 128 of the C2 model (bench.py's configuration, bf16, eval mode) trained on an analytic
    sphere of radius 1 (white background) with its 128^3 occupancy grid, measured after each number of steps in
    `checkpoints` (the longer the training, the more opaque the surface): reference-semantics render_image, chunked
    render_rays with the grid, and b2n.render_image_fast at t_min = 0 and 1e-4.  Medians over 10 runs after 3 warm-ups.
    After the last checkpoint the wave budget (b2n.render.WAVE_POINTS) is swept at t_min = 1e-4."""
    import subprocess
    from b2n import render as br
    from b2n import synthetic
    from src.renderer import DensityGrid, render_image, render_rays
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                # noqa: BLE001 -- the measurement stands without it
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, power.max_limit: {smi}")
    sys.path.insert(0, ROOT)
    from bench import C2, GRID_R, GRID_THR
    near, far, radius = 2.0, 6.0, 1.0
    b2n.set_mlp_precision("bf16")
    torch.manual_seed(0)
    model = NeuralField(C2).cuda().train()
    grid = DensityGrid(resolution=GRID_R, bound=C2["scene_bound"], threshold=GRID_THR).cuda()
    opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-5)
    bg = torch.ones(3, device="cuda")
    ro, rd = synthetic.image_rays(synthetic.hemisphere_poses(1, seed=123)[0], H=H, W=H)
    ro, rd = ro.cuda(), rd.cuda()
    rays = H * H

    def sphere(o, d):
        b = (o * d).sum(-1)
        disc = b * b - ((o * o).sum(-1) - radius ** 2)
        p = o + d * (-b - torch.sqrt(disc.clamp_min(0)))[:, None]
        col = torch.stack([0.5 + 0.5 * p[:, 2], 0.2 + 0.3 * p[:, 0], 0.5 - 0.5 * p[:, 2]], -1).clamp(0, 1)
        return torch.where((disc > 0)[:, None], col, torch.ones_like(col))

    def image():
        return render_image(model, ro.view(H, H, 3), rd.view(H, H, 3), near, far, N, chunk, True)

    def masked():
        outs = [render_rays(model, ro[i:i + chunk], rd[i:i + chunk], near, far, N, False, density_grid=grid)
                for i in range(0, rays, chunk)]
        return [torch.cat(x) for x in zip(*outs)]

    def fast(t_min):
        return br.render_image_fast(model, ro.view(H, H, 3), rd.view(H, H, 3), near, far, N, density_grid=grid,
                                    t_min=t_min)

    step = 0
    for stop in checkpoints:
        model.train()
        for step in range(step + 1, stop + 1):
            o, d, _ = (t.cuda() for t in synthetic.random_rays(2 ** 16, seed=step))
            pred, _, _ = render_rays(model, o, d, near, far, 64, True, density_grid=grid, bg_color=bg)
            loss = torch.nn.functional.mse_loss(pred, sphere(o, d))
            opt.zero_grad()
            loss.backward()
            opt.step()
            if step >= 50 and step % 16 == 0:
                model.eval()
                grid.update(model, device="cuda")
                model.train()
        model.eval()
        occ = grid.update(model, device="cuda")
        with torch.no_grad():
            psnr = -10 * torch.log10(((image().view(-1, 3) - sphere(ro, rd)) ** 2).mean())
            ref = masked()
            n_masked = b2n.march.march(ro, rd, near, far, N, None, bits=grid.bits(), R=grid.resolution,
                                       bound=grid.bound).n_active
            print(f"\nC2 trained {stop} steps on a sphere of radius {radius}: loss {loss.item():.5f}, grid occupancy "
                  f"{occ:.3f}, test-view PSNR {psnr.item():.2f} dB; view {H}x{H}, N={N}, wave budget 2^"
                  f"{br.WAVE_POINTS.bit_length() - 1}")
            legs = [("render_image (reference semantics, every sample)", image, rays * N, None),
                    ("render_rays with the grid, chunks of 2^16 rays", masked, n_masked, None),
                    ("render_image_fast t_min=0", lambda: fast(0.0), None, 0.0),
                    ("render_image_fast t_min=1e-4", lambda: fast(1e-4), None, 1e-4)]
            for name, fn, n_eval, t_min in legs:
                med, best = timeit(fn, n=10, warm=3)
                extra = ""
                if t_min is not None:
                    out = fast(t_min)
                    n_eval = out.n_evaluated
                    err = [float((a.reshape(b.shape) - b).abs().max()) for a, b in zip(out[:3], ref)]
                    extra = (f", {out.n_waves} waves, max |diff| to the masked path: color {err[0]:.2e} "
                             f"depth {err[1]:.2e} acc {err[2]:.2e}")
                print(f"{name}: median {med:.3f} ms (best {best:.3f}), {n_eval / rays:.2f} evaluated samples per ray"
                      f"{extra}")
            out = br.render_image_fast(model, ro.view(H, H, 3), rd.view(H, H, 3), near, far, N, density_grid=grid,
                                       t_min=1e-4, _samples_per_wave=1)
            print(f"composited samples per ray at t_min=1e-4 (one sample per wave): {out.n_evaluated / rays:.2f}")
    default = br.WAVE_POINTS
    try:
        with torch.no_grad():
            for wp in (2 ** 18, 2 ** 19, 2 ** 20, 2 ** 21, 2 ** 22, 2 ** 23, 2 ** 24):
                br.WAVE_POINTS = wp
                med, best = timeit(lambda: fast(1e-4), n=10, warm=3)
                out = fast(1e-4)
                print(f"wave budget 2^{wp.bit_length() - 1}: t_min=1e-4 median {med:.3f} ms (best {best:.3f}), "
                      f"{out.n_waves} waves, {out.n_evaluated / rays:.2f} evaluated samples per ray")
    finally:
        br.WAVE_POINTS = default


def _device_line():
    import subprocess
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:                                # noqa: BLE001 -- the measurement stands without it
        smi = f"nvidia-smi unavailable ({e})"
    print(f"device: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, power.max_limit: {smi}")


def _torch_importance(sigma, z, rd, Nf, U):
    """the rule of b2n_importance_sample as torch ops (cumprod, cumsum, searchsorted, gather, stable sort)"""
    B, Nc = z.shape
    delta = torch.cat([z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], 1e10)], -1) * rd.norm(dim=-1, keepdim=True)
    alpha = -torch.expm1(-sigma * delta)
    w = alpha * torch.cumprod(torch.cat([torch.ones_like(alpha[:, :1]), 1.0 - alpha[:, :-1] + 1e-10], -1), -1)
    mids = 0.5 * (z[:, 1:] + z[:, :-1])
    wi = w[:, 1:-1] + 1e-5
    cdf = torch.cat([torch.zeros_like(wi[:, :1]), torch.cumsum(wi / wi.sum(-1, keepdim=True), -1)], -1)
    u = (torch.arange(Nf, device=z.device) + U) / Nf
    i = torch.searchsorted(cdf, u, right=True)
    below, above = (i - 1).clamp_min(0), i.clamp_max(Nc - 2)
    cb, ca = torch.gather(cdf, 1, below), torch.gather(cdf, 1, above)
    mb, ma = torch.gather(mids, 1, below), torch.gather(mids, 1, above)
    denom = ca - cb
    denom = torch.where(denom < 1e-5, torch.ones_like(denom), denom)
    zf = mb + (u - cb) / denom * (ma - mb)
    zm, src = torch.sort(torch.cat([z, zf], -1), dim=-1, stable=True)
    return zf, zm, src


def importance(Nc=64, Nf=128, quality_steps=1000):
    """Hierarchical sampling (b2n.importance, DESIGN.md §5h): (1) the sampler kernel against the same rule as torch ops
    at the C1 batch (B = 4096, L2-resident) and one 800^2 view (640 000 rays), in HBM bytes/s of the algorithmic
    traffic; (2) a C1 training step (vanilla model, bf16, B = 4096) with 64 + 128 hierarchical samples against
    stratified N = 64 and N = 192, and the cost of the merged-order gather inside it; (3) held-out PSNR on the analytic
    spheres of tests/test_gpu_training.py after a fixed number of steps: hierarchical 64 + 128 against stratified
    N = 192 (as many composited samples) and N = 256 (NeRF's evaluation count)."""
    from b2n import march, synthetic
    from b2n.importance import _gather, importance_sample, render_rays_hierarchical
    from src.renderer import render_rays
    _device_line()
    torch.manual_seed(0)
    # (1) the sampler
    for B in (4096, 640_000):
        ro, rd, _ = (t.cuda() for t in synthetic.random_rays(B, seed=1))
        z = march.march(ro, rd, 2.0, 6.0, Nc, torch.rand(B, Nc, device="cuda")).z
        sigma = torch.rand(B, Nc, device="cuda") * 4 * (torch.rand(B, Nc, device="cuda") < 0.5)
        U = torch.rand(B, Nf, device="cuda")
        nbytes = B * (8.0 * Nc + 12 + 4.0 * Nf + 4.0 * Nf + 8.0 * (Nc + Nf))
        ours = importance_sample(sigma, z, rd, Nf, U)
        ref = _torch_importance(sigma, z, rd, Nf, U)
        dz = float((ours[0] - ref[0]).abs().max())
        same_src = float((ours[2].long() == ref[2]).float().mean())
        for name, fn in (("b2n_importance_sample", lambda: importance_sample(sigma, z, rd, Nf, U)),
                         ("torch ops", lambda: _torch_importance(sigma, z, rd, Nf, U))):
            med, best = timeit(fn, n=20, warm=3)
            print(f"sampler B={B} {Nc}+{Nf} [{name}]: median {med:.4f} ms (best {best:.4f}), "
                  f"{nbytes / med / 1e6:.0f} GB/s of the kernel's {nbytes / B:.0f} B/ray")
        print(f"  kernel vs torch ops: max |dz_fine| {dz:.2e}, merge sources equal for {100 * same_src:.3f} % of slots")
    # (2) the C1 step
    b2n.set_mlp_precision("bf16")
    B = 4096
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(B, seed=1))
    for leg in ("stratified N=64", "stratified N=192", f"hierarchical {Nc}+{Nf}"):
        torch.manual_seed(0)
        model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().train()
        opt = torch.optim.Adam(model.parameters(), lr=5e-4)
        tgt = torch.rand(B, 3, device="cuda")

        def step():
            if leg.startswith("hier"):
                out = render_rays_hierarchical(model, ro, rd, 2.0, 6.0, Nc, Nf, True)
                loss = torch.nn.functional.mse_loss(out.color, tgt) + torch.nn.functional.mse_loss(out.coarse_color, tgt)
            else:
                pred = render_rays(model, ro, rd, 2.0, 6.0, int(leg.split("=")[1]), True, white_bkgd=True)[0]
                loss = torch.nn.functional.mse_loss(pred, tgt)
            opt.zero_grad()
            loss.backward()
            opt.step()
        med, best = timeit(step, n=20, warm=3)
        print(f"C1 train step [bf16] B={B} {leg}: median {med:.3f} ms (best {best:.3f})")
    M = Nc + Nf
    idx = torch.sort(torch.rand(B, M, device="cuda"), -1).indices
    rgb_c = torch.rand(B * Nc, 3, device="cuda", requires_grad=True)
    rgb_f = torch.rand(B * Nf, 3, device="cuda", requires_grad=True)
    s_c = torch.rand(B * Nc, 1, device="cuda", requires_grad=True)
    s_f = torch.rand(B * Nf, 1, device="cuda", requires_grad=True)

    def gather():
        out = _gather(rgb_c, rgb_f, idx).sum() + _gather(s_c, s_f, idx).sum()
        torch.autograd.grad(out, [rgb_c, rgb_f, s_c, s_f])
    med, best = timeit(gather, n=20, warm=3)
    print(f"merged-order gather of rgb + sigma, forward + backward, B={B} {Nc}+{Nf}: median {med:.3f} ms")
    # (3) quality at a fixed step budget
    for radius, lr in ((0.6, 5e-4), (1.2, 1e-3)):
        def sphere(o, d):
            b = (o * d).sum(-1)
            disc = b * b - ((o * o).sum(-1) - radius ** 2)
            n = (o + d * (-b - torch.sqrt(disc.clamp_min(0)))[:, None]) / radius
            col = torch.stack([0.5 + 0.5 * n[:, 2], 0.2 + 0.0 * n[:, 0], 0.5 - 0.5 * n[:, 2]], -1)
            return torch.where((disc > 0)[:, None], col, torch.ones_like(col))
        held_o, held_d, _ = (t.cuda() for t in synthetic.random_rays(16384, seed=9999))
        held_t = sphere(held_o, held_d)
        for leg in (f"hierarchical {Nc}+{Nf}", "stratified N=192", "stratified N=256"):
            torch.manual_seed(0)
            model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().train()
            opt = torch.optim.Adam(model.parameters(), lr=lr)
            hier = leg.startswith("hier")
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for step in range(1, quality_steps + 1):
                o, d, _ = (t.cuda() for t in synthetic.random_rays(2048, seed=step))
                tgt = sphere(o, d)
                if hier:
                    out = render_rays_hierarchical(model, o, d, 2.0, 6.0, Nc, Nf, True)
                    loss = torch.nn.functional.mse_loss(out.color, tgt) + torch.nn.functional.mse_loss(out.coarse_color, tgt)
                else:
                    pred = render_rays(model, o, d, 2.0, 6.0, int(leg.split("=")[1]), True, white_bkgd=True)[0]
                    loss = torch.nn.functional.mse_loss(pred, tgt)
                opt.zero_grad()
                loss.backward()
                opt.step()
            e1.record()
            torch.cuda.synchronize()
            model.eval()
            with torch.no_grad():
                if hier:
                    out = render_rays_hierarchical(model, held_o, held_d, 2.0, 6.0, Nc, Nf, False)
                    pred, coarse = out.color, out.coarse_color
                else:
                    pred = render_rays(model, held_o, held_d, 2.0, 6.0, int(leg.split("=")[1]), False)[0]
                    coarse = None
            psnr = -10 * torch.log10(((pred - held_t) ** 2).mean()).item()
            extra = "" if coarse is None else f" (its coarse pass alone: {-10 * torch.log10(((coarse - held_t) ** 2).mean()).item():.2f} dB)"
            print(f"sphere r={radius}, {quality_steps} steps of 2048 rays, Adam lr={lr}, {leg}: held-out PSNR {psnr:.2f} dB"
                  f"{extra}, training {e0.elapsed_time(e1) / quality_steps:.3f} ms/step")
    b2n.check_errors()


def _band_scene(ro, rd, radius=0.6, band=0.25):
    """the checker-band sphere of tests/test_gpu_errormap.py: a shaded sphere with a 24 x 6 black-and-white checker on
    the latitude band |n_z| < band, white background; returns (colour [B,3], on-band mask [B])"""
    b = (ro * rd).sum(-1)
    disc = b * b - ((ro * ro).sum(-1) - radius ** 2)
    hit = disc > 0
    n = (ro + rd * (-b - torch.sqrt(disc.clamp_min(0)))[:, None]) / radius
    col = torch.stack([0.5 + 0.5 * n[:, 2], 0.2 + 0.0 * n[:, 0], 0.5 - 0.5 * n[:, 2]], -1)
    on = hit & (n[:, 2].abs() < band)
    az = torch.atan2(n[:, 1], n[:, 0])
    check = ((torch.floor(az * 24 / (2 * 3.141592653589793)) + torch.floor(n[:, 2] * 6 / (2 * band))) % 2)
    col = torch.where(on[:, None], check[:, None].expand(-1, 3), col)
    return torch.where(hit[:, None], col, torch.ones_like(col)), on


def errormap(steps=2000, B_train=8192):
    """Error-map sampling (b2n.errormap, DESIGN.md §5i): (1) sample + update at the C2 size (2^18 rays, 100 views of
    800^2, 128^2 cells per view) against the 21.5 ms C2 step; (2) held-out PSNR after a fixed number of steps on the
    checker-band sphere, Instant model, uniform picks against the error map at uniform_frac = 0.25 (unweighted loss,
    as Instant-NGP), with the step time of each leg: PSNR over every training pixel (what the sampler spends its rays
    on) and over held-out views."""
    from b2n import synthetic
    from b2n.errormap import ErrorMap
    from src.renderer import render_rays
    _device_line()
    # (1) the sampler at C2 size, the map filled by a few updates first (an all-unobserved map samples uniformly)
    V, H, W, B = 100, 800, 800, 2 ** 18
    emap = ErrorMap(V, H, W)
    gen = torch.Generator(device="cuda").manual_seed(0)
    for _ in range(20):
        picks, _ = emap.sample(B, generator=gen)
        emap.update(picks, torch.rand(B, device="cuda", generator=gen))
    picks, _ = emap.sample(B, generator=gen)
    err = torch.rand(B, device="cuda", generator=gen)
    n = emap.cdf.numel()
    print(f"map {V} x {H} x {W}, cells {emap.Hm} x {emap.Wm} ({n} cells, CDF {n * 8 / 1e6:.1f} MB), B = {B}; "
          f"{int((emap.e >= 0).sum())} cells observed")
    t_s, b_s = timeit(lambda: emap.sample(B, generator=gen), n=50, warm=5)
    t_u, b_u = timeit(lambda: emap.update(picks, err), n=50, warm=5)
    t_c, _ = timeit(emap.rebuild_cdf, n=50, warm=5)

    def both():
        p, _ = emap.sample(B, generator=gen)
        emap.update(p, err)
    t_b, b_b = timeit(both, n=50, warm=5)
    print(f"sample (torch.rand + 1 kernel): median {t_s:.4f} ms (best {b_s:.4f})")
    print(f"update (accumulate + apply + CDF, 5 kernels): median {t_u:.4f} ms (best {b_u:.4f}); of it the CDF "
          f"rebuild alone {t_c:.4f} ms ({n * 16 / t_c / 1e6:.0f} GB/s of its {n * 16 / 1e6:.1f} MB)")
    print(f"sample + update: median {t_b:.4f} ms (best {b_b:.4f}) = {100 * t_b / 21.5:.2f} % of the 21.5 ms C2 step")
    # (2) quality at a fixed step budget on the checker-band sphere
    b2n.set_mlp_precision("bf16")
    Vt, Ht = 100, 128
    cfg = dict(mode="part2_instant", n_levels=12, n_features_per_level=2, log2_hashmap_size=17, base_resolution=16,
               per_level_scale=1.5, scene_bound=1.5, L_embed_dir=4, hidden_dim=64)

    def views(nv, seed):
        poses = synthetic.hemisphere_poses(nv, seed=seed)
        ro, rd = zip(*(synthetic.image_rays(p, H=Ht, W=Ht) for p in poses))
        ro, rd = torch.stack(ro).cuda(), torch.stack(rd).cuda()
        tgt, on = _band_scene(ro.reshape(-1, 3), rd.reshape(-1, 3))
        return ro, rd, tgt.reshape(nv, Ht * Ht, 3), on
    tr_o, tr_d, tr_t, tr_on = views(Vt, 21)
    he_o, he_d, he_t, he_on = views(8, 22)
    bg = torch.ones(3, device="cuda")

    def psnr(model, o, d, t, on):
        o, d, t = o.reshape(-1, 3), d.reshape(-1, 3), t.reshape(-1, 3)
        with torch.no_grad():
            pred = torch.cat([render_rays(model, o[i:i + 2 ** 15], d[i:i + 2 ** 15], 2.0, 6.0, 64, False,
                                          bg_color=bg)[0] for i in range(0, o.shape[0], 2 ** 15)])
        mse = ((pred - t) ** 2).mean(-1)
        return -10 * torch.log10(mse.mean()).item(), -10 * torch.log10(mse[on].mean()).item()
    for leg in ("uniform", "error map, uniform_frac=0.25"):
        torch.manual_seed(0)
        model = NeuralField(cfg).cuda().train()
        opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=1e-5)
        em = ErrorMap(Vt, Ht, Ht, cells=(32, 32), uniform_frac=0.25)
        g = torch.Generator(device="cuda").manual_seed(1)
        use_map = leg.startswith("error")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            if use_map:
                (v, y, x), _ = em.sample(B_train, generator=g)
            else:
                v, y, x = (torch.randint(0, k, (B_train,), device="cuda", generator=g) for k in (Vt, Ht, Ht))
            k = y * Ht + x
            pred = render_rays(model, tr_o[v, k], tr_d[v, k], 2.0, 6.0, 64, True, bg_color=bg)[0]
            per_ray = ((pred - tr_t[v, k]) ** 2).mean(-1)
            opt.zero_grad()
            per_ray.mean().backward()
            opt.step()
            if use_map:
                em.update((v, y, x), per_ray.detach())
        e1.record()
        torch.cuda.synchronize()
        model.eval()
        fit, fit_band = psnr(model, tr_o, tr_d, tr_t, tr_on)
        held, held_band = psnr(model, he_o, he_d, he_t, he_on)
        print(f"checker-band sphere, {Vt} views of {Ht}^2, {steps} steps of {B_train} rays, Instant model, {leg}: "
              f"PSNR over all training pixels {fit:.2f} dB (band {fit_band:.2f}), held-out {held:.2f} dB "
              f"(band {held_band:.2f}), {e0.elapsed_time(e1) / steps:.3f} ms/step")
    b2n.check_errors()


def c1_step(P_rays=4096, N=64):
    """C1: vanilla NeRF training step (render_rays + MSE + backward + Adam), B=4096, N=64."""
    from b2n import synthetic
    from src.renderer import render_rays
    for mode in ("bf16", "fp32"):
        b2n.set_mlp_precision(mode)
        torch.manual_seed(0)
        model = NeuralField(dict(mode="part2_nerf", L_embed=10, L_embed_dir=4)).cuda().train()
        opt = torch.optim.Adam(model.parameters(), lr=5e-4)
        ro, rd, tgt = (t.cuda() for t in synthetic.random_rays(P_rays, seed=1))

        def step():
            pred, _, _ = render_rays(model, ro, rd, 2.0, 6.0, N, True, white_bkgd=True)
            loss = torch.nn.functional.mse_loss(pred, tgt[:, :3])
            opt.zero_grad()
            loss.backward()
            opt.step()

        med, best = timeit(step, n=5 if mode == "fp32" else 20, warm=3)
        if mode == "bf16" and "--prof" in sys.argv:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    step()
                torch.cuda.synchronize()
            print(prof.key_averages().table(sort_by="cuda_time_total", row_limit=25, max_name_column_width=60))
        flops = 3 * 2.0 * P_rays * N * 593408
        print(f"C1 train step [{mode}] B={P_rays} N={N}: median {med:.3f} ms -> {P_rays / med * 1e3 / 1e6:.3f} M rays/s, "
              f"{flops / med / 1e9:.1f} TFLOP/s algorithmic")
        model.eval()
        with torch.no_grad():
            med, best = timeit(lambda: render_rays(model, ro, rd, 2.0, 6.0, N, False, white_bkgd=True), n=10, warm=2)
        print(f"C1 render [{mode}]: median {med:.3f} ms -> {P_rays * N / med * 1e3 / 1e6:.1f} Msamples/s")


def hash_levels(P=24_000_000):
    """hash fwd / bwd time as a function of the level range (contention study)."""
    from b2n import synthetic, march
    torch.manual_seed(0)
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(2 ** 18, seed=1))
    u = torch.rand(2 ** 18, 128, device="cuda")
    occ = torch.ones(128, 128, 128, dtype=torch.bool, device="cuda")
    m = march.march(ro, rd, 2.0, 6.0, 128, u, bits=march.pack_occupancy(occ), R=128, bound=1.5)
    x = m.pts
    print("points", x.shape[0])
    for (nl, base, note) in ((16, 16, "all 16 levels"), (4, 16, "levels 0-3 (dense 16..54)"), (8, 16, "levels 0-7"),
                             (4, 411, "4 fine hashed levels (res 411..1384)")):
        geom = b2n.HashGeometry(nl, base, 1.5, 19, 2)
        table = torch.randn(geom.n_params, device="cuda", requires_grad=True) * 0.1
        table = table.detach().requires_grad_(True)
        y = b2n.hash_encode(x, table, geom, 1.5)
        g = torch.randn_like(y)
        f_med, _ = timeit(lambda: b2n.hash_encode(x, table, geom, 1.5), n=5, warm=2)

        def bwd():
            y = b2n.hash_encode(x, table, geom, 1.5)
            y.backward(g)
        b_med, _ = timeit(bwd, n=5, warm=2)
        print(f"{note:45s} L={nl:2d}: fwd {f_med:7.3f} ms ({f_med / nl:6.3f}/level)  bwd(+fwd+memset) {b_med - f_med:7.3f} ms "
              f"({(b_med - f_med) / nl:6.3f}/level)")


def hash_sorted():
    """The spatially ordered hash-grid path of the C2 step (dense occupancy, 2^18 rays x 128 samples, L = 16, F = 2,
    T = 2^19): hash_encode forward + backward as the C2 step runs it (b2n_hash_order, b2n_hash_fwd_ordered,
    b2n_hash_bwd_ordered), with the table gradient's warp-level entry merge on the levels with res <= dedup_res
    (b2n_debug_hash_dedup; 0 = run merging up to res 128), the settings alternated; then the table-gradient scatter
    alone per 4-level window [lbeg, lbeg + 4) for each setting.  Per entry: median (best) of 10 calls, CUDA events.
    Result: profiles/hashdedup_b200.txt, DESIGN.md section 7b."""
    from b2n import synthetic, march
    _device_line()
    torch.manual_seed(0)
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(2 ** 18, seed=1))
    u = torch.rand(2 ** 18, 128, device="cuda")
    occ = torch.ones(128, 128, 128, dtype=torch.bool, device="cuda")
    x = march.march(ro, rd, 2.0, 6.0, 128, u, bits=march.pack_occupancy(occ), R=128, bound=1.5).pts
    P = x.shape[0]
    geom = b2n.HashGeometry(16, 16, 1.5, 19, 2)
    print("points", P, "| level res:", " ".join(str(lv[1]) for lv in geom.levels))
    table = (torch.randn(geom.n_params, device="cuda") * 0.1).requires_grad_(True)
    settings = (0, 54, 81, 122, 183, 274, 616, 1 << 20)
    keys = ("b2n_hash_order", "b2n_hash_fwd", "b2n_hash_bwd")
    g = None
    times = {d: {k: [] for k in keys} for d in settings}
    for rep in range(10):
        for d in settings:                                    # alternated: each setting sees the same clocks
            with _lib.hash_dedup(d):
                y = b2n.hash_encode(x, table, geom, 1.5)
                if g is None:
                    g = torch.randn_like(y)
                table.grad = None
                torch.cuda.synchronize()
                _lib.PROFILER = prof = _lib.Profiler()
                y = b2n.hash_encode(x, table, geom, 1.5)
                y.backward(g)
                torch.cuda.synchronize()
                _lib.PROFILER = None
            for n_, _, _, e0, e1 in prof.records:
                if n_ in times[d]:
                    times[d][n_].append(e0.elapsed_time(e1))
    for d in settings:
        ts = {k: sorted(v) for k, v in times[d].items()}
        med = {k: v[len(v) // 2] for k, v in ts.items()}
        print(f"hash_encode fwd+bwd dedup_res={d:7d}: " + ", ".join(f"{k} {med[k]:.3f} ({ts[k][0]:.3f})" for k in keys)
              + f" ms, sum {sum(med.values()):.3f} ms")

    order = torch.empty(P, dtype=torch.int32, device="cuda")
    xs = torch.empty_like(x)
    scratch = torch.empty(_lib.lib.b2n_hash_order_scratch(P) // 4, dtype=torch.int32, device="cuda")
    _lib.call("b2n_hash_order", _lib.ptr(x), P, 1.5, _lib.ptr(order), _lib.ptr(xs), _lib.ptr(scratch), _lib.stream())
    G = torch.zeros(geom.n_params, device="cuda")
    L = geom.n_levels
    for lbeg in range(0, L, 4):
        def scatter():
            _lib.call("b2n_hash_bwd_ordered", _lib.ptr(xs), _lib.ptr(order), P, 1.5, _lib.ptr(table), geom.c_levels, L, 2,
                      _lib.ptr(g), 2 * L, 0, _lib.ptr(G), lbeg, lbeg + 4, _lib.stream())
        res = [geom.levels[l][1] for l in range(lbeg, lbeg + 4)]
        ts = {d: [] for d in settings}
        for rep in range(10):
            for d in settings:
                with _lib.hash_dedup(d):
                    ts[d].append(timeit(scatter, n=1, warm=1)[0])
        print(f"scatter levels [{lbeg:2d}, {lbeg + 4:2d}) res {res}: " +
              ", ".join(f"dedup_res={d} {sorted(v)[len(v) // 2]:.3f} ({min(v):.3f})" for d, v in ts.items()) + " ms")


def hash_variants():
    """A/B of the F = 2 hash-grid kernels on the C2 sample set (24 M active points, L = 16, T = 2^19) and the C5 canonical
    geometry (T = 2^20): (point, level)-per-lane kernels against the pair-lane kernels, and the run-merging threshold."""
    from b2n import synthetic, march
    hash_variant = b2n._lib.hash_variant
    torch.manual_seed(0)
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(2 ** 18, seed=1))
    u = torch.rand(2 ** 18, 128, device="cuda")
    occ = torch.ones(128, 128, 128, dtype=torch.bool, device="cuda")
    x = march.march(ro, rd, 2.0, 6.0, 128, u, bits=march.pack_occupancy(occ), R=128, bound=1.5).pts
    print("points", x.shape[0])
    for log2T in (19, 20):
        geom = b2n.HashGeometry(16, 16, 1.5, log2T, 2)
        table = (torch.randn(geom.n_params, device="cuda") * 0.1).requires_grad_(True)
        with hash_variant(0, 64):
            y_ref = b2n.hash_encode(x, table, geom, 1.5)
            g = torch.randn_like(y_ref)
            gt_ref, = torch.autograd.grad((y_ref * g).sum(), table)
        for variant, merge in ((0, 64), (1, 64), (2, 0), (2, 24), (2, 64), (2, 128), (2, 200), (3, 64), (3, 128)):
            with hash_variant(variant, merge):
                y = b2n.hash_encode(x, table, geom, 1.5)
                gt, = torch.autograd.grad((y * g).sum(), table)
                ey = float((y - y_ref).abs().max() / y_ref.abs().max())
                eg = float((gt - gt_ref).abs().max() / gt_ref.abs().max())
                b2n._lib.PROFILER = prof = b2n._lib.Profiler()
                for _ in range(4):
                    y = b2n.hash_encode(x, table, geom, 1.5)
                    y.backward(g)
                torch.cuda.synchronize()
                b2n._lib.PROFILER = None
            print(f"T=2^{log2T} variant={variant} merge_res={merge:3d}: " +
                  ", ".join(f"{k} {min(e0.elapsed_time(e1) for n_, _, _, e0, e1 in prof.records if n_ == k):.3f} ms"
                            for k in ("b2n_hash_fwd", "b2n_hash_bwd")) + f"   max rel diff vs variant 0: y {ey:.2e} g_table {eg:.2e}")


def red_bench():
    """red.global.add throughput on an L2-resident table: per lane or per sector?"""
    from b2n._lib import call, ptr, stream
    names = {0: "v2 random lanes", 1: "v2 lane pairs share 16 B", 2: "v2 4 lanes share a sector", 3: "v4 random lanes",
             4: "v4 even lanes only", 5: "v2 even lanes only", 6: "v2 16 lanes share a 128-B line"}
    for log2n in (18, 22):
        n = 1 << log2n
        table = torch.zeros(n, 2, device="cuda")
        blocks, per_thread = 148 * 16, 256
        for mode in range(7):
            fn = lambda: call("b2n_debug_red_bench", ptr(table), n, blocks, per_thread, mode, stream())
            med, best = timeit(fn, n=5, warm=2)
            lanes = blocks * 256 * per_thread * (0.5 if mode in (4, 5) else 1.0)
            print(f"table {n * 8 >> 20:3d} MiB mode {mode} ({names[mode]:32s}): {lanes / best / 1e6:8.1f} G lane-ops/s, "
                  f"{blocks * 8 * per_thread / best / 1e6:7.2f} G warp-instr/s")


def l2_gather():
    """Random 8-byte gathers over tables of 2 MiB .. 512 MiB: the L2 (and beyond-L2) gather peak."""
    from b2n._lib import call, ptr, stream
    sink = torch.zeros(1, device="cuda")
    out = {}
    for log2n in (18, 21, 22, 23, 24, 26):          # float2 entries: 2 MiB, 16, 32, 64, 128, 512 MiB
        n = 1 << log2n
        table = torch.randn(n, 2, device="cuda")
        blocks, per_thread = 148 * 16, 512
        fn = lambda: call("b2n_debug_gather_bench", ptr(table), n, blocks, per_thread, ptr(sink), stream())
        med, best = timeit(fn, n=5, warm=2)
        g = blocks * 256 * per_thread
        out[n * 8 >> 20] = g / best / 1e6
        print(f"table {n * 8 >> 20:4d} MiB: {g / best / 1e6:8.1f} G gathers/s  = {g * 8 / best / 1e6:7.1f} GB/s useful, "
              f"{g * 32 / best / 1e6:7.1f} GB/s of 32-byte sectors")
    return out


def composite(B=2 ** 18, N=128):
    """compositing forward / backward on the C2 shapes: dense occupancy (~72 % of samples active, compact layout)"""
    from b2n import synthetic, march
    torch.manual_seed(0)
    ro, rd, _ = (t.cuda() for t in synthetic.random_rays(B, seed=1))
    u = torch.rand(B, N, device="cuda")
    for kind in ("dense", "sparse"):
        occ = torch.ones(128, 128, 128, dtype=torch.bool, device="cuda") if kind == "dense" else synthetic.ball_occupancy(128, 1.5).cuda()
        m = march.march(ro, rd, 2.0, 6.0, N, u, bits=march.pack_occupancy(occ), R=128, bound=1.5)
        Pn = m.pts.shape[0]
        rgb = torch.rand(Pn, 3, device="cuda", requires_grad=True)
        sigma = (torch.rand(Pn, device="cuda") * 2).requires_grad_(True)
        bg = torch.ones(3, device="cuda")
        from b2n import _lib
        g = torch.randn(B, 3, device="cuda")

        def both():
            c, d, a, _ = b2n.composite(rgb, sigma, m.z, rd, bg=bg, mask_words=m.mask_words, ray_offset=m.ray_offset)
            torch.autograd.grad((c * g).sum(), [rgb, sigma])
        for _ in range(3):
            both()
        torch.cuda.synchronize()
        prof = _lib.Profiler()
        _lib.PROFILER = prof
        for _ in range(20):
            both()
        torch.cuda.synchronize()
        _lib.PROFILER = None
        for name, v in prof.summary().items():
            print(f"composite [{kind}] B={B} N={N} active={Pn}: {name} {v['ms'] / v['calls']:.4f} ms = "
                  f"{v['bytes'] / v['ms'] / 1e6:.0f} GB/s algorithmic ({100 * v['bytes'] / v['ms'] / 1e6 / 6496.8:.1f} % of measured HBM peak)")


def mlp64(P=1 << 22):
    """fused Instant decoder: forward (1 or 2 point tiles in flight per CTA) and backward (1 or 3 warp groups per CTA),
    C2-sized (4.2 M points) and Part-3 width"""
    from oracle import nerf_oracle as O
    for pos_dim in (32, 53):
        gen = torch.Generator().manual_seed(0)
        sp = O._fused_init(pos_dim, 16, 64, 1, gen).cuda().requires_grad_(True)
        cp = O._fused_init(43, 3, 64, 2, gen).cuda().requires_grad_(True)
        x = (torch.randn(P, pos_dim, device="cuda") * 0.5).requires_grad_(True)
        d = torch.nn.functional.normalize(torch.randn(P, 3, device="cuda"), dim=-1)
        bands = O.fourier_bands(4).cuda()
        for slots in (1, 2):
            _lib.lib.b2n_debug_instant_fwd_slots(slots)
            with torch.no_grad():
                med, best = timeit(lambda: b2n.instant_mlp(x, d, bands, sp, cp))
                meds, bests = timeit(lambda: b2n.instant_sigma(x, sp))
            print(f"instant fwd pos_dim={pos_dim} P={P} slots={slots}: {med:.3f} ms (best {best:.3f}); sigma-only {meds:.3f} ms")
        b2n.check_errors()
        rgb, sigma = b2n.instant_mlp(x, d, bands, sp, cp)
        g1, g2 = torch.randn_like(rgb), torch.randn_like(sigma)
        for groups in (1, 3):
            _lib.lib.b2n_debug_instant_bwd_groups(groups)
            med, best = timeit(lambda: torch.autograd.grad([rgb, sigma], [x, sp, cp], [g1, g2], retain_graph=True))
            print(f"instant bwd pos_dim={pos_dim} P={P} groups={groups}: {med:.3f} ms (best {best:.3f})")
        b2n.check_errors()


def overlap(P=12_000_000):
    """can the L2-atomic-bound table scatter and the SM-bound decoder backward share the SMs?  Independent inputs, two streams."""
    from oracle import nerf_oracle as O
    from src.embeddings import HashGridEncoding
    gen = torch.Generator().manual_seed(0)
    sp = O._fused_init(32, 16, 64, 1, gen).cuda().requires_grad_(True)
    cp = O._fused_init(43, 3, 64, 2, gen).cuda().requires_grad_(True)
    x = (torch.randn(P, 32, device="cuda") * 0.5).requires_grad_(True)
    d = torch.nn.functional.normalize(torch.randn(P, 3, device="cuda"), dim=-1)
    bands = O.fourier_bands(4).cuda()
    # autograd runs a backward node on the stream of its forward: issue each forward on the stream its backward should use
    s1, s2 = torch.cuda.Stream(priority=-1), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        rgb, sigma = b2n.instant_mlp(x, d, bands, sp, cp)
        g1, g2 = torch.randn_like(rgb), torch.randn_like(sigma)
    enc = HashGridEncoding(3, dict(otype="HashGrid", n_levels=16, n_features_per_level=2, log2_hashmap_size=19,
                                   base_resolution=16, per_level_scale=1.5)).cuda()
    # ray-ordered samples like the training step: 128 samples along random rays
    B = P // 128
    o = (torch.rand(B, 1, 3, device="cuda") - 0.5) * 2
    dd = torch.nn.functional.normalize(torch.randn(B, 1, 3, device="cuda"), dim=-1)
    tt = torch.linspace(0, 2.0, 128, device="cuda").view(1, 128, 1)
    pts = ((o + dd * tt).reshape(-1, 3).clamp(-1.5, 1.5) / 3.0 + 0.5).contiguous()          # unit cube
    torch.cuda.synchronize()
    with torch.cuda.stream(s2):
        feat = enc(pts)
        gf = torch.randn_like(feat)
    torch.cuda.synchronize()

    def mlp():
        torch.autograd.grad([rgb, sigma], [x, sp, cp], [g1, g2], retain_graph=True)

    def hashb():
        torch.autograd.grad(feat, enc.params, gf, retain_graph=True)

    def both():
        cur = torch.cuda.current_stream()
        s1.wait_stream(cur), s2.wait_stream(cur)
        with torch.cuda.stream(s1):
            mlp()
        with torch.cuda.stream(s2):
            hashb()
        cur.wait_stream(s1), cur.wait_stream(s2)

    for groups in (3, 1, 4):
        _lib.lib.b2n_debug_instant_bwd_groups(groups)
        tm, _ = timeit(mlp)
        th, _ = timeit(hashb)
        tb, _ = timeit(both)
        print(f"groups={groups}: decoder bwd {tm:.3f} ms, table scatter {th:.3f} ms, both on two streams {tb:.3f} ms (sum {tm + th:.3f})")
    _lib.lib.b2n_debug_instant_bwd_groups(3)


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "mlp256"
    P = int(sys.argv[2]) if len(sys.argv) > 2 and sys.argv[2].isdigit() else 262144
    if what == "c1":
        c1_step()
    elif what == "occ":
        occ_update()
    elif what == "mesh":
        mesh()
    elif what == "render":
        render()
    elif what == "importance":
        importance()
    elif what == "errormap":
        errormap()
    elif what == "hashsort":
        hash_sorted()
    elif what == "hash":
        hash_levels()
    elif what == "hashv":
        hash_variants()
    elif what == "red":
        red_bench()
    elif what == "l2":
        l2_gather()
    elif what == "overlap":
        overlap()
    elif what == "mlp64":
        mlp64()
    elif what == "composite":
        composite()
        composite(8192, 64)
    else:
        {"mlp256": mlp256, "mlp256x": mlp256x, "mlp256t": mlp256t}[what](P)
