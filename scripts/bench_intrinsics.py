"""Cost of per-image camera intrinsics and of the intrinsics gradients in the fused view-synthesis loss.

Three cases of the same md2_view_synthesis_loss_fwdbwd step (the one bench.py times), alternated in one process:
  (a) shared K, no K gradient          -- the call as it was before intrinsics became per image / differentiable
  (b) per-image K, no K gradient
  (c) per-image K with grad_K and grad_invK
The per-image K of (b) and (c) are N copies of the shared camera of (a): every case then warps the same pixels, and the
differences are the cost of the per-image camera path and of the intrinsics gradients, not of a different geometry.
at config 2 (416x128x8, C=1) and config 3 (640x192x12, C=3, automask formed inside the call).  Each case is timed with
CUDA events over a ring of input sets larger than the L2 (like bench.py), in several alternating rounds, and reports
steps/s (median over rounds), the spread over rounds and kernel launches per step.  One JSON line per (config, case);
the GPU's name and power limit are read in the same run.

    python scripts/bench_intrinsics.py [--steps 400] [--warmup 20] [--rounds 5]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import monodepth2_jl_b200 as M                          # noqa: E402
from monodepth2_jl_b200 import _lib as L                # noqa: E402
from monodepth2_jl_b200 import synthetic as SY          # noqa: E402

CONFIGS = {2: (8, 1, 128, 416, False), 3: (12, 3, 192, 640, True)}
SCALES = (0.125, 0.25, 0.5, 1.0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 else (torch.cuda.get_device_name(), "?")
    return name, power


def run_config(cfg, args, dev, ctx):
    N, Cc, H, W, am = CONFIGS[cfg]
    g = torch.Generator().manual_seed(7)
    K, invK = SY.make_K(W, H)
    Kp, iKp = K.expand(N, 3, 3), invK.expand(N, 3, 3)
    cm = lambda m: m.transpose(-1, -2).contiguous().to(dev)
    intr = {"a": (cm(K), cm(invK), False, False), "b": (cm(Kp), cm(iKp), True, False), "c": (cm(Kp), cm(iKp), True, True)}
    set_bytes = 4 * N * 3 * Cc * H * W * 2
    n_sets = max(4, int(2.5 * 126e6 / set_bytes) + 1)
    sets = []
    for k in range(n_sets):
        x = torch.rand(N, 3, Cc, H, W, generator=g).to(dev)
        disps = [torch.rand(N, 1, max(2, round(H * s)), max(2, round(W * s)), generator=g).to(dev) for s in SCALES]
        rv = [(0.01 * torch.randn(N, 3, generator=g)).to(dev) for _ in range(2)]
        tv = [(0.01 * torch.randn(N, 3, generator=g)).to(dev) for _ in range(2)]
        sets.append(dict(x=x, disps=disps, rv=rv, tv=tv, loss=torch.zeros((), device=dev), gd=[torch.empty_like(d) for d in disps],
                         gr=[torch.empty_like(r) for r in rv], gt=[torch.empty_like(t) for t in tv], gx=torch.empty_like(x)))
    descs = {}
    for case, (Kc, iKc, per, grad) in intr.items():
        gK, giK = (torch.empty_like(Kc), torch.empty_like(iKc)) if grad else (None, None)
        descs[case] = [L.make_vsl_desc(
            target=st["x"][:, 1], target_stride=st["x"].stride(0), sources=[st["x"][:, 0], st["x"][:, 2]],
            source_strides=[st["x"].stride(0)] * 2, disparities=st["disps"], K_cm=Kc, invK_cm=iKc, per_image_K=per,
            grad_K=gK, grad_invK=giK, rot=st["rv"], trans=st["tv"], pose_mode=1, invert=[1, 0], compute_automask=am,
            smooth_weight=[1e-3 * s for s in SCALES], loss_scale=1.0 / len(SCALES), loss=st["loss"], grad_disparity=st["gd"],
            grad_rot=st["gr"], grad_trans=st["gt"], grad_source=[st["gx"][:, 0], st["gx"][:, 2]], zero_grad_source=True,
            shape=(N, Cc, H, W)) for st in sets]
        descs[case].append((gK, giK))
    lib, handle = ctx.lib, ctx.handle
    stream = torch.cuda.current_stream(dev)
    sptr = stream.cuda_stream

    def step(case, i):
        if lib.md2_view_synthesis_loss_fwdbwd(handle, C.byref(descs[case][i % n_sets]), 1.0, sptr):
            raise RuntimeError(lib.md2_last_error().decode())

    for case in intr:   # warm-up: every ring slot twice (first sighting eager, second captures the graph), then W more
        for i in range(2 * n_sets + args.warmup):
            step(case, i)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = {c: [] for c in intr}
    launches = {}
    for r in range(args.rounds):
        for case in (intr if r % 2 == 0 else list(intr)[::-1]):
            l0 = ctx.launches
            e0.record(stream)
            for i in range(args.steps):
                step(case, i)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            res[case].append(args.steps / (e0.elapsed_time(e1) * 1e-3))
            launches[case] = (ctx.launches - l0) / args.steps
    med = {c: sorted(v)[len(v) // 2] for c, v in res.items()}
    name, power = gpu_info()
    for case in intr:
        v = res[case]
        print(json.dumps({"config": cfg, "shape": f"{W}x{H}x{N} C={Cc}" + (" automask" if am else ""), "case": case,
                          "per_image_K": intr[case][2], "grad_K": intr[case][3], "steps_per_s": round(med[case], 1),
                          "spread_steps_per_s": [round(min(v), 1), round(max(v), 1)], "launches_per_step": launches[case],
                          "us_per_step_over_a": round(1e6 / med[case] - 1e6 / med["a"], 2), "gpu": name, "power_limit": power,
                          "steps": args.steps, "rounds": args.rounds}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--config", type=int, nargs="*", default=[2, 3])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_intrinsics.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ctx = M.Context.get(dev)
    for cfg in args.config:
        run_config(cfg, args, dev, ctx)


if __name__ == "__main__":
    main()
