"""bench.py contract checks that need no GPU: the reference arm (the reference's CPU implementation of the training
step -- the real reference + tcnn shim when /root/reference exists, else the oracle port) prints ONE well-formed JSON
line, and the product arm refuses to run without CUDA (there is no CPU fallback to measure by accident)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, **env_overrides):
    env = dict(os.environ, OMP_NUM_THREADS="4", **env_overrides)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env,
                          timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-rays", "64")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_rays_per_s" and d["unit"] == "rays/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_refuses_to_run_without_cuda():
    # no device visible to the child process, also on a machine that has one
    r = _run("--steps", "1", "--warmup", "0", "--no-extras", "--no-cpu-baseline", CUDA_VISIBLE_DEVICES="")
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout)
