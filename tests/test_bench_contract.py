"""bench.py's contract on a machine without a GPU: the reference arm (the oracle port of the reference's CPU path) prints one JSON
line with the keys the driver reads; the product arm refuses to run (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None and d["dtype"] == "f32"
    assert d["config"]["workload"].startswith("configs[1]: 416x128, batch 8/GPU")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert cb["value_1_thread"] > 0 and cb["value_c_oracle_f64_1_thread"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_refuses_to_run_without_a_gpu():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)
    assert not any(l.startswith("{") for l in r.stdout.splitlines())


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_step(tmp_path):
    """--dump-outputs: float32 .npy files of at most 64 MB in all, holding the loss and gradients of the last timed step; with
    --steps 1 that step ran on the first ring slot, the package's seeded batch, so the oracle can recompute it"""
    from monodepth2_jl_b200 import synthetic as SY
    from util import check_vsl_statistical, oracle_vsl
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1", "--no-cpu-baseline",
                        "--no-train-step", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][0])["steps"] == 1
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == sorted(["loss"] + [f"grad_disparity_{l}" for l in range(4)] +
                                 [f"grad_{k}_{s}" for k in ("rot", "trans", "source") for s in range(2)])
    assert all(a.dtype == np.float32 for a in got.values()) and sum(a.nbytes for a in got.values()) <= 64 << 20
    x, disps, rv, tv = SY.synthetic_batch(8, 1, 128, 416, seed=42)
    K, invK = SY.make_K(416, 128)
    ref = oracle_vsl(x, disps, rv, tv, K, invK)
    t = lambda k: torch.from_numpy(got[k])
    gx = torch.zeros_like(x)
    gx[:, 0], gx[:, 2] = t("grad_source_0"), t("grad_source_1")
    out = dict(loss=float(got["loss"]), gdisp=[t(f"grad_disparity_{l}") for l in range(4)], grvec=[t("grad_rot_0"), t("grad_rot_1")],
               gtvec=[t("grad_trans_0"), t("grad_trans_1")], gx=gx)
    check_vsl_statistical(out, ref, tag="bench --dump-outputs")
