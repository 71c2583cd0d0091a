"""bench.py on the GPU: --steps sets the number of timed headline steps, and --dump-outputs writes what the LAST of them
computed (float32 .npy files, large arrays as a fixed 2^20-element sample) from inputs that are the same in every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
RAYS = 4096
PARAMS = ("representation.encoding.params", "decoder.sigma_net.params", "decoder.color_net.params")


def _bench(steps, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--rays", str(RAYS),
           "--no-extras", "--no-cpu-baseline"] + (["--dump-outputs", str(dump)] if dump else [])
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == steps
    return d, ({f[:-4]: np.load(dump / f) for f in os.listdir(dump)} if dump else None)


def _rel_l2(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-30))


def test_steps_and_dump_outputs(tmp_path):
    d1, _ = _bench(1)
    d2, a = _bench(2, tmp_path / "a")
    _, b = _bench(2, tmp_path / "b")
    # every timed step launches the same kernels: twice the steps, twice the launches in the timed region
    assert d1["gpu_launches"] > 0 and d2["gpu_launches"] == 2 * d1["gpu_launches"]

    assert set(a) == {"color", "depth", "acc", "loss"} | {f"{k}.{p}" for k in ("param", "grad") for p in PARAMS}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert a["color"].shape == (RAYS, 3) and a["depth"].shape == (RAYS,) and a["acc"].shape == (RAYS,)
    assert a["loss"].shape == ()
    assert a["param.representation.encoding.params"].shape == (2 ** 20,)       # sample of the 13 M-entry table
    assert a["grad.decoder.color_net.params"].shape == a["param.decoder.color_net.params"].shape == (8192,)
    assert float(np.abs(a["grad.representation.encoding.params"]).max()) > 0
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) < 64 * 2 ** 20

    # color and loss are those of the last timed step: the warm-up step renders batch 0, timed step i batch i % 3 and
    # the later e2e leg ends on batch 2, so with 2 timed steps the loss is the MSE of the color against batch 1
    # (the TV term adds ~1e-8)
    from b2n import synthetic
    mse = []
    for i in range(3):
        rgba = synthetic.random_rays(RAYS, seed=i)[2].numpy().astype(np.float64)
        target = rgba[:, :3] * rgba[:, 3:4] + (1.0 - rgba[:, 3:4])
        mse.append(float(np.mean((a["color"] - target) ** 2)))
    assert abs(mse[1] - float(a["loss"])) < 1e-4 * float(a["loss"]), (mse, float(a["loss"]))
    assert min(abs(mse[0] - mse[1]), abs(mse[2] - mse[1])) > 1e-3 * mse[1], mse

    # same inputs and same sampled table positions in both runs: only atomics-order noise between them
    for name in a:
        assert _rel_l2(a[name], b[name]) < (1e-2 if name.startswith(("param.", "grad.")) else 1e-3), name
