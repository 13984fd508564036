#!/usr/bin/env python
"""Benchmark of the hot path: the fused view-synthesis loss (warp + SSIM/L1 photometric loss,
forward + backward, all 4 decoder scales) of Monodepth2.jl training.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference --gpus N --steps K    # the reference's CPU path (oracle port)
  python bench.py --steps K --dump-outputs DIR           # also write the last timed step's loss and gradients (DIR/*.npy)

A "step" is one pass of the hot path over one synthetic batch.  Workload at every N:
BASELINE.json configs[1] -- 416x128, batch 8 per GPU, C=1 (KITTI gray as in train()),
S=2 sources, 4 scales at the decoder's native sizes, no automask, gradients to the
disparities, the poses and the source images (g=1 of BASELINE.md's work model).
Inputs are resident in HBM before the timed region; the steps rotate through a ring of
input/gradient sets larger than twice the L2, so no step finds its inputs in cache.
One JSON line on stdout (rank 0).
"""
import argparse
import ctypes as C
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

W_, H_, NB, CH, S_, LS = 416, 128, 8, 1, 2, 4
AM = False
SCALES = (0.125, 0.25, 0.5, 1.0)
METRIC = "train frames/s @416x128 R18: view-synthesis loss path (warp + SSIM/L1 loss, fwd+bwd, 4 scales)"
WORKLOAD = "configs[1]: 416x128, batch 8/GPU, C=1, S=2, L=4 native-size disparities, no automask, g=1"
# BASELINE.json configs reachable with --config (default 2 = configs[1], the one the metric is quoted on)
CONFIGS = {
    2: dict(W=416, H=128, N=8, C=1, am=False, name="configs[1]: 416x128, batch 8/GPU, C=1, S=2, L=4 native-size disparities, no automask, g=1"),
    3: dict(W=640, H=192, N=12, C=3, am=True, name="configs[2]: 640x192, batch 12/GPU, C=3, S=2, L=4 native-size disparities, automask + min-reprojection, g=1"),
    4: dict(W=1024, H=320, N=4, C=3, am=False, name="configs[3]: 1024x320, batch 4/GPU, C=3, S=2, L=4 native-size disparities, no automask, g=1"),
}


def set_config(k):
    global W_, H_, NB, CH, AM, WORKLOAD, METRIC
    c = CONFIGS[k]
    W_, H_, NB, CH, AM, WORKLOAD = c["W"], c["H"], c["N"], c["C"], c["am"], c["name"]
    METRIC = f"train frames/s @{W_}x{H_} R18: view-synthesis loss path (warp + SSIM/L1 loss, fwd+bwd, 4 scales)"


def algorithmic_bytes(W, H, N, C, S, L, m=0, g=1):
    """BASELINE.md section 3: fwd 4(1+C+SC+m) + bwd 4(1+C+SC+m) + 4(1+gSC) bytes per unit"""
    per_unit = 4 * (1 + C + S * C + m) * 2 + 4 * (1 + g * S * C)
    return per_unit * W * H * N * L, per_unit


def ncu_static():
    """per-launch figures of the dominant kernel that only a profiler can see (one `ncu --set full` capture of this very
    command, committed under profiles/): DRAM bytes and executed warp instructions"""
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    return json.load(open(tp)) if os.path.exists(tp) else {}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def bind_to_gpu_cpus(index):
    """pin this process to the CPUs NVML reports as local to the GPU (its NUMA node), so that the pinned host
    buffers are allocated there and host<->device copies do not cross the socket interconnect"""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n = (os.cpu_count() + 63) // 64
        masks = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = {64 * i + b for i, m in enumerate(masks) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class ClockSampler(threading.Thread):
    """polls NVML for SM clock and throttle reasons while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.stop_flag, self.max_mhz = [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def sample(self):
        if not self.nv:
            return
        nv = self.nv
        try:
            self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
                     0x4: "sw_power_cap", 0x80: "hw_power_brake"}
            for bit, name in names.items():
                if r & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def run(self):
        # (a query every 10 ms: NVML calls take a driver-wide lock, and eight ranks polling every 2 ms showed up as launch jitter)
        while not self.stop_flag:
            self.sample()
            time.sleep(0.010)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def make_sets(n_sets, dev, seed0, smooth=False):
    """ring of independent input + gradient-output sets, each built from the package's seeded
    synthetic generator (monodepth2_jl_b200.synthetic; the tests check that it produces exactly
    the data of the oracle-side generator).
    smooth=True: disparities as a depth network produces them -- smooth fields (a coarse random field, bilinearly
    enlarged, the same scene at every scale) instead of the generator's low-passed noise with +-10 % per-pixel jitter per ring
    slot.  The warp of a smooth disparity samples neighbouring cells for neighbouring pixels (coalesced gathers and
    reductions); the noisy default scatters them over ~14 sectors per warp instruction and is the harsher case."""
    from monodepth2_jl_b200 import synthetic as SY
    base = SY.synthetic_batch(NB, CH, H_, W_, seed=seed0)
    sets = []
    g = torch.Generator().manual_seed(seed0 + 1)
    for i in range(n_sets):
        x, disps, rv, tv = base
        if smooth:
            coarse = torch.randn(NB, 1, max(2, H_ // 32), max(2, W_ // 32), generator=g)
            disps = [torch.sigmoid(1.5 * torch.nn.functional.interpolate(coarse, size=tuple(d.shape[-2:]), mode="bilinear", align_corners=True)).contiguous()
                     for d in disps]
            if i:
                x = (x + 0.02 * torch.rand(x.shape, generator=g)).clamp(0, 1)
        elif i:   # cheap decorrelated variants of the base batch (different data per ring slot)
            x = (x + 0.02 * torch.rand(x.shape, generator=g)).clamp(0, 1)
            disps = [(d * (0.9 + 0.2 * torch.rand(d.shape, generator=g))).clamp(0.01, 0.99) for d in disps]
        sets.append(dict(
            x=x.to(dev), disps=[d.to(dev) for d in disps], rv=[r.to(dev) for r in rv], tv=[t.to(dev) for t in tv],
            loss=torch.zeros((), device=dev), gd=[torch.empty_like(d, device=dev) for d in disps],
            gr=[torch.empty(NB, 3, device=dev) for _ in range(S_)], gt=[torch.empty(NB, 3, device=dev) for _ in range(S_)],
            gx=torch.zeros(x.shape, device=dev), am=None))
    return sets, base


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, st, grad_x):
    """writes what md2_view_synthesis_loss_fwdbwd handed back for the input set `st` as float32 DIR/<name>.npy, named after
    the md2_vsl_desc fields: loss, grad_disparity_<scale>, grad_rot_<source>, grad_trans_<source>, grad_source_<source>
    (the inputs are seeded, so two builds run with the same arguments can be compared output for output)"""
    import numpy as np
    arrays = {"loss": st["loss"]}
    arrays.update({f"grad_disparity_{l}": g for l, g in enumerate(st["gd"])})
    for s, frame in enumerate((0, 2)):      # the source frames of desc_for
        arrays[f"grad_rot_{s}"], arrays[f"grad_trans_{s}"] = st["gr"][s], st["gt"][s]
        if grad_x:
            arrays[f"grad_source_{s}"] = st["gx"][:, frame]
    host = {k: v.float().cpu().numpy() for k, v in arrays.items()}
    nbytes = sum(a.nbytes for a in host.values())
    if nbytes > DUMP_MAX_BYTES:
        raise SystemExit(f"--dump-outputs: {nbytes} B of outputs exceed the {DUMP_MAX_BYTES} B limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    print(f"wrote {len(host)} outputs ({nbytes / 1e6:.1f} MB) to {out_dir}", file=sys.stderr)


def run_ours(args):
    import monodepth2_jl_b200 as M
    from monodepth2_jl_b200 import _lib as L
    from monodepth2_jl_b200 import synthetic as SY

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    all_cpus = os.sched_getaffinity(0)
    bound = bind_to_gpu_cpus(local) if not args.no_bind else None   # pinned buffers + launches from the GPU's NUMA node
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout when the communicator is created: keep stdout for the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    ctx = M.Context.get(dev)
    ctx_sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
    K, invK = SY.make_K(W_, H_)
    K_cm, invK_cm = K.t().contiguous().to(dev), invK.t().contiguous().to(dev)
    sw = [1e-3 * s for s in SCALES]

    abytes, per_unit = algorithmic_bytes(W_, H_, NB, CH, S_, LS, m=1 if AM else 0)
    l2_bytes = 126e6
    set_bytes = 4 * (NB * 3 * CH * H_ * W_ * 2 + 2 * sum(int(NB * round(H_ * s) * round(W_ * s)) for s in SCALES))
    n_sets = max(4, int(2.5 * l2_bytes / set_bytes) + 1)
    sets, base = make_sets(n_sets, dev, 42 + rank)
    # (automasking: the map is formed INSIDE the timed call, desc.compute_automask -- the per-step pre-pass of src/Monodepth.jl:159-164)
    grad_x = not os.environ.get("MD2_BENCH_G0")

    def desc_for(st):
        x = st["x"]
        return L.make_vsl_desc(
            target=x[:, 1], target_stride=x.stride(0), sources=[x[:, 0], x[:, 2]], source_strides=[x.stride(0)] * 2,
            disparities=st["disps"], K_cm=K_cm, invK_cm=invK_cm, rot=st["rv"], trans=st["tv"], pose_mode=1,
            invert=[1, 0], automask=None, compute_automask=AM, smooth_weight=sw, loss_scale=1.0 / LS, normalize_disparity=True, loss=st["loss"],
            grad_disparity=st["gd"], grad_rot=st["gr"], grad_trans=st["gt"],
            grad_source=([st["gx"][:, 0], st["gx"][:, 2]] if grad_x else None), zero_grad_source=True, shape=(NB, CH, H_, W_))

    descs = [desc_for(st) for st in sets]
    lib, handle = ctx.lib, ctx.handle
    stream = torch.cuda.current_stream(dev)
    sptr = stream.cuda_stream
    fwdbwd = lib.md2_view_synthesis_loss_fwdbwd

    def step(i):
        # (the source-image gradient is accumulated with atomics: desc.zero_grad_source makes the
        # library's prep kernel zero-fill it, so a step is exactly one C-ABI call)
        rc = fwdbwd(handle, C.byref(descs[i % n_sets]), 1.0, sptr)
        if rc:
            raise RuntimeError(lib.md2_last_error().decode())

    def barrier():
        if dist:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # warm-up: at least W steps, and enough to bring clocks up and touch every ring slot
    warm = max(args.warmup, 3, n_sets)
    t0 = time.time()
    k = 0
    while k < warm or time.time() - t0 < 0.3:
        step(k)
        k += 1
    barrier()

    sampler = ClockSampler(local)
    sampler.sample()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ctx.launches
    barrier()
    e0.record(stream)
    for i in range(args.steps):
        step(i)
    e1.record(stream)
    barrier()
    sampler.sample()
    sampler.stop_flag = True
    launches = ctx.launches - l0
    if args.dump_outputs and rank == 0:
        # (now: the sections below run the same ring slots again and overwrite their outputs)
        dump_outputs(args.dump_outputs, sets[(args.steps - 1) % n_sets], grad_x)
    from monodepth2_jl_b200 import dist as D
    ms = D.max_over_ranks(e0.elapsed_time(e1), device=dev)   # device time, max over ranks
    frames = NB * world * args.steps
    value = frames / (ms * 1e-3)

    # ---- the same call warm (one input set back to back: L2-resident) and forward-only (cold ring), SURVEY 8(d) ----
    def timed(fn, n):
        for i in range(2 * n_sets + 2):      # (every descriptor of the ring twice: first sighting eager, second captures its graph)
            fn(i)
        barrier()
        e0.record(stream)
        for i in range(n):
            fn(i)
        e1.record(stream)
        barrier()
        return D.max_over_ranks(e0.elapsed_time(e1), device=dev) / n
    fwd_only = lib.md2_view_synthesis_loss_fwd

    def step_fwd(i):
        if fwd_only(handle, C.byref(descs[i % n_sets]), sptr):
            raise RuntimeError(lib.md2_last_error().decode())
    n_var = min(args.steps, 500)
    variants = {"fwdbwd_warm_l2_ms": round(timed(lambda i: step(0), n_var), 5), "fwd_only_cold_ms": round(timed(step_fwd, n_var), 5),
                "fwd_only_warm_l2_ms": round(timed(lambda i: step_fwd(0), n_var), 5),
                "note": "same workload; warm = one input set back to back (L2-resident), cold = the ring; fwd_only = md2_view_synthesis_loss_fwd (loss value only)"}

    # ---- the same workload on smooth disparities (what a depth network produces), cold ring: step and marching kernel ----
    sets_s, _ = make_sets(n_sets, dev, 4242 + rank, smooth=True)
    descs_s = [desc_for(st) for st in sets_s]

    def step_s(i):
        if fwdbwd(handle, C.byref(descs_s[i % n_sets]), 1.0, sptr):
            raise RuntimeError(lib.md2_last_error().decode())
    for i in range(2 * n_sets + 2):
        step_s(i)
    variants["fwdbwd_smooth_disparity_ms"] = round(timed(step_s, n_var), 5)
    ctx.profile(True)
    for i in range(n_var):
        step_s(i)
    sk, sn = ctx.profile_read()
    ctx.profile(False)
    variants["march_kernel_smooth_disparity_ms"] = round(sk / max(sn, 1), 5)
    variants["smooth_note"] = ("smooth disparities = a coarse random field bilinearly enlarged (same scene at every scale), as a depth network produces them; "
                               "the headline workload keeps the generator's noisy disparities (neighbouring pixels sample cells several pixels apart), the harsher case")
    del sets_s, descs_s

    # ---- roofline of the dominant kernel: second pass with per-launch CUDA events ----
    ctx.profile(True)
    for i in range(args.steps):
        step(i)
    kms, kn = ctx.profile_read()
    ctx.profile(2)          # time stamps around all three launches (serialises them: no programmatic overlap)
    for i in range(min(args.steps, 500)):
        step(i)
    pa, pb, pc, pn = ctx.profile_read_phases()
    ctx.profile(False)
    phases = {"prep_us": round(1e3 * pa / max(pn, 1), 2), "march_us": round(1e3 * pb / max(pn, 1), 2), "finish_us": round(1e3 * pc / max(pn, 1), 2),
              "note": "CUDA events between the three launches of a step (warm, in the pipeline); the event records add to the gaps between the launches, "
                      "so the sum exceeds ms_per_step"}
    k_ms = kms / max(kn, 1)
    peak, peak_src = peaks()
    achieved = abytes / (k_ms * 1e-3) / 1e9
    ncu = ncu_static() if (CH, AM, NB, W_) == (1, False, 8, 416) else {}     # (the committed capture is of the default workload)
    traffic = ncu.get("fused_bwd_c1_bytes_per_launch")
    # instruction roofline of the same kernel (it is issue-bound, not memory-bound): executed warp instructions per launch
    # (ncu: smsp__inst_executed.sum) against one instruction per scheduler and clock on every SM sub-partition
    issue = None
    if ncu.get("march_warp_insts_per_launch"):
        sm_clock = 1e6 * (sampler.summary()["sm_mhz"] or 1965)
        floor_ms = ncu["march_warp_insts_per_launch"] / (ctx_sm_count * 4 * sm_clock) * 1e3
        issue = {"warp_insts_per_launch": ncu["march_warp_insts_per_launch"], "lane_insts_per_unit": round(32.0 * ncu["march_warp_insts_per_launch"] / (abytes / per_unit), 1),
                 "floor_ms": round(floor_ms, 5), "frac": round(floor_ms / k_ms, 4), "unit": "issue slots (1 warp instruction per scheduler per clock)",
                 "source": ncu.get("source")}

    # ---- e2e: host-buffer entry point (md2_view_synthesis_loss_fwdbwd_host through the package's
    # HostViewSynthesisLoss): every step copies the batch from pinned host memory to the device, runs the
    # kernels and copies the loss and all gradients back; the call is synchronous (it returns when the host
    # buffers hold the results), so the steps are timed back to back on the host clock ----
    hx, hd, hr, ht = base
    Kd, invKd = K.to(dev), invK.to(dev)
    h_am = None
    import gc

    def time_host(grad_x, e_steps, lanes=1):
        """lanes = 1: synchronous calls back to back (each returns when its results are in host memory);
        lanes = 2: double-buffered -- step i+1 is submitted on the other lane before step i is collected, so a step's
        device-to-host copies overlap the next step's host-to-device copies and kernels.  Every step still moves its own
        inputs from pinned host memory and its own results back; the loop collects every step's loss."""
        # (image groups overlap copies and kernels INSIDE a call; with two lanes the overlap comes from the next call)
        hv = M.HostViewSynthesisLoss(NB, CH, H_, W_, [(d.shape[-1], d.shape[-2]) for d in hd], K, invK, device=dev,
                                     scales=SCALES, groups=args.e2e_groups if lanes == 1 else 1, grad_x=grad_x, automask="inside" if AM else False, lanes=lanes)
        for lane in range(lanes):
            hv.fill(lane, hx, hd, hr, ht, automask=h_am)
        if lanes == 1:
            run = lambda: hv()
            hv()                                # first call sizes the workspaces and captures the graph
        else:
            for lane in range(lanes):           # (captures every lane's graph)
                hv.submit(lane)
            hv.wait(0)
            state = {"k": 0}

            def run():                          # one step: submit on the free lane, collect the OLDEST step in flight
                lane = state["k"] % lanes
                hv.submit(lane)
                state["k"] += 1
                return hv.wait((lane + 1) % lanes)
        for _ in range(6):
            run()
        barrier()
        gc.collect()
        gc.disable()
        per_call = []
        t0 = time.perf_counter()
        for _ in range(e_steps):
            t1 = time.perf_counter()
            run()
            per_call.append(time.perf_counter() - t1)
        if lanes > 1:
            for j in range(1, lanes):           # the steps still in flight
                hv.wait((state["k"] - j) % lanes)
        e_ms = D.max_over_ranks((time.perf_counter() - t0) * 1e3, device=dev)
        gc.enable()
        per_call.sort()
        pct = [round(per_call[min(len(per_call) - 1, int(q / 100 * len(per_call)))] * 1e3, 4) for q in (5, 50, 95)]
        barrier()
        return NB * world * e_steps / (e_ms * 1e-3), e_ms, pct, hv.h2d_bytes, hv.d2h_bytes

    def pcie_probe(h2d_bytes, d2h_bytes):
        """the floor of the end-to-end step on THIS box at THIS N: the step's bytes at the best rate the host link shows
        in this run with all ranks copying at once (pinned buffers of 64 MB, 16 MB and of the step's own size, back to
        back, each direction; the host->device rate of these boxes varies with the transfer size, so the best is taken)"""
        rates = {"h2d": 0.0, "d2h": 0.0}
        for nbytes in (64 << 20, 16 << 20, h2d_bytes):
            n = nbytes // 4
            hbuf, dbuf = torch.empty(n).pin_memory(), torch.empty(n, device=dev)
            for direction in ("h2d", "d2h"):
                def burst(k):
                    for _ in range(k):
                        (dbuf.copy_(hbuf, non_blocking=True) if direction == "h2d" else hbuf.copy_(dbuf, non_blocking=True))
                    torch.cuda.synchronize(dev)
                burst(3)
                barrier()
                t0 = time.perf_counter()
                burst(8)
                ms = D.max_over_ranks((time.perf_counter() - t0) * 1e3, device=dev) / 8
                rates[direction] = max(rates[direction], 4 * n / (ms * 1e-3) / 1e9)
                barrier()
        return max(h2d_bytes / rates["h2d"], d2h_bytes / rates["d2h"]) / 1e6, rates, (h2d_bytes / rates["h2d"] + d2h_bytes / rates["d2h"]) / 1e6

    e_steps = min(args.steps, 500)
    # what a training step needs on the host: the loss and the gradients of the network outputs (disparities, poses).
    # The gradient of the source IMAGES (g = 1 of the device-resident figure) is computed by Zygote in the reference and
    # thrown away -- it is not an output a trainer reads back; the same call with it copied back too is `value_g1`.
    e2e_sync, es_ms, es_pct, h2d, d2h = time_host(False, e_steps, lanes=1)
    e2e_value, e_ms, e2e_pct, _, _ = time_host(False, e_steps, lanes=args.e2e_lanes)
    e2e_g1, _, _, h2d_g1, d2h_g1 = time_host(True, max(50, e_steps // 2), lanes=args.e2e_lanes)
    floor_ms, link, floor_shared_ms = pcie_probe(h2d, d2h)

    # the same through the autograd mirror of the reference API (torch tensors, many small copies): secondary figure
    pin = lambda t: t.contiguous().pin_memory()
    px, pd, pr_, pt = pin(hx), [pin(d) for d in hd], [pin(r) for r in hr], [pin(t) for t in ht]
    dx = torch.empty_like(px, device=dev)
    dd = [torch.empty_like(d, device=dev).requires_grad_(True) for d in pd]
    dr = [torch.empty_like(r, device=dev).requires_grad_(True) for r in pr_]
    dt = [torch.empty_like(t, device=dev).requires_grad_(True) for t in pt]
    h_loss = torch.zeros((), pin_memory=True)
    h_gd = [torch.empty_like(d).pin_memory() for d in pd]
    h_gp = [torch.empty(NB, 3).pin_memory() for _ in range(2 * S_)]

    def e2e_step():
        dx.copy_(px, non_blocking=True)
        with torch.no_grad():
            for a, b in zip(dd + dr + dt, pd + pr_ + pt):
                a.copy_(b, non_blocking=True)
        for a in dd + dr + dt:
            a.grad = None
        loss = M.view_synthesis_loss(dx, dd, dr, dt, Kd, invKd, K_cm=K_cm, invK_cm=invK_cm, compute_automask=AM)
        loss.backward()
        h_loss.copy_(loss.detach(), non_blocking=True)
        for a, b in zip(h_gd + h_gp, dd + dr + dt):
            a.copy_(b.grad, non_blocking=True)
        torch.cuda.synchronize(dev)   # the caller consumes the host results every step

    for _ in range(5):
        e2e_step()
    barrier()
    a_steps = min(args.steps, 200)
    e0.record(stream)
    for _ in range(a_steps):
        e2e_step()
    e1.record(stream)
    barrier()
    a_ms = D.max_over_ranks(e0.elapsed_time(e1), device=dev)
    e2e_autograd = NB * world * a_steps / (a_ms * 1e-3)

    out = {
        "metric": METRIC, "value": round(value, 1), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": round(ms / args.steps, 5), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded KITTI-shaped triplets, random-init poses/disparities)",
        "config": {"workload": WORKLOAD, "width": W_, "height": H_, "batch_per_gpu": NB, "channels": CH,
                   "sources": S_, "scales": LS, "automask": AM, "automask_map": "formed inside the timed call (desc.compute_automask)" if AM else None,
                   "grad_source_images": True,
                   "l2_policy": f"inputs larger than L2: ring of {n_sets} input/gradient sets ({n_sets * set_bytes / 1e6:.0f} MB) rotated per step",
                   "api": "md2_view_synthesis_loss_fwdbwd (C ABI), one call per step", "sharding": "batch, no data-path collective"},
        "images_per_s": round(3 * value, 1),
        "variants": variants,
        "gpu_launches": int(launches),
        "clocks": sampler.summary(),
        # (the headline is the better of the two ways of driving the same entry point: with several ranks on one host the
        # host's memory / PCIe path saturates and keeping more steps in flight only adds contention)
        "e2e": {"value": round(max(e2e_value, e2e_sync), 1), "mode": "multi-buffered (value_multi_buffered)" if e2e_value >= e2e_sync else "synchronous calls (value_synchronous)",
                "unit": "frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "value_multi_buffered": round(e2e_value, 1),
                "steps": e_steps, "ms_per_step": round(min(e_ms, es_ms) / e_steps, 5), "ms_per_step_multi_buffered": round(e_ms / e_steps, 5), "ms_per_call_p5_p50_p95": e2e_pct,
                "grad_source_images": False,
                "note": "host outputs = loss + disparity / pose gradients (g=0: the source-image gradient, which the reference's training loop "
                        "discards, is neither formed nor copied back); value_g1 = the same call with the source-image gradients formed and copied back too",
                "value_g1": round(e2e_g1, 1), "d2h_bytes_per_step_g1": d2h_g1,
                "api": "md2_view_synthesis_loss_fwdbwd_host_submit / md2_host_wait (C ABI, host pointers; copies and kernels of a call on "
                       "copy/compute streams, replayed as a CUDA graph; " + f"{args.e2e_lanes} lanes: a step is submitted before the oldest one in flight is collected; the pinned inputs / gradients of a lane are one "
                       "allocation each and travel as one copy each way) via monodepth2_jl_b200.HostViewSynthesisLoss, every step's loss and gradients collected on the host",
                "value_synchronous": round(e2e_sync, 1), "ms_per_step_synchronous": round(es_ms / e_steps, 5), "ms_per_call_synchronous_p5_p50_p95": es_pct,
                "pcie_floor_ms": round(floor_ms, 5), "pcie_floor_frames_per_s": round(NB * world / (floor_ms * 1e-3), 1),
                "pcie_floor_ms_if_directions_share_the_host_path": round(floor_shared_ms, 5),
                "host_link_GBps_per_gpu": {k: round(v, 1) for k, v in link.items()},
                "pcie_floor_note": f"the step's {h2d} B host->device and {d2h} B device->host at the best rate the host link showed in this run "
                                   f"(pinned copies of 64 MB / 16 MB / the step's size, all {world} rank(s) at once, one direction at a time): max of the two directions "
                                   "(full duplex: what one GPU sees); their sum is the floor when the ranks saturate a shared host path (what eight GPUs see)",
                "autograd_api_value": round(e2e_autograd, 1), "cpus_bound_to_gpu_numa_node": bound},
        "roofline": {"bound": "hbm", "kernel": f"march2_kernel<C={CH},S=2,AM={int(AM)}> (fused fwd+bwd single-warp marching kernel, all scales in one launch)",
                     "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                     "traffic": traffic, "algorithmic_bytes_per_launch": abytes, "bytes_per_unit": per_unit,
                     "kernel_ms": round(k_ms, 5), "kernel_launches_timed": int(kn), "peak_source": peak_src,
                     "step_frac_of_peak": round(abytes / (ms / args.steps * 1e-3) / 1e9 / peak, 4), "issue_roofline": issue, "step_phases": phases},
    }
    if not args.no_train_step:
        out["train_step"] = train_step_bench(args, dev, rank, world, dist, barrier)
    if args.train_step:      # the whole training step as the main line (second metric; the loss path stays under "loss_path")
        ts = out["train_step"]
        out["loss_path"] = {k: out[k] for k in ("metric", "value", "unit", "ms_per_step", "gpu_launches")}
        out.update(metric=f"train frames/s @{W_}x{H_} R18 stand-in: full data-parallel training step", value=ts["value"], ms_per_step=ts["ms_per_step"],
                   steps=ts["steps"], warmup=ts["warmup"], gpu_launches=ts["md2_launches"])
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)   # the CPU arm gets every host core
            out["cpu_baseline"] = cpu_baseline(base, budget_s=15.0)
        print(json.dumps(out), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def train_step_bench(args, dev, rank, world, dist, barrier):
    """Row F1: the reference's training step (src/Monodepth.jl:156-176) as a data-parallel step -- stand-in R18 encoder +
    depth / pose decoders on the host framework's conv layers (not part of this library), THIS library's fused loss
    (train_loss), backward, the parameter-gradient all-reduce over NCCL in buckets overlapped with backward, one fused
    ADAM launch.  Timed with CUDA events, max over ranks; at N > 1 also without the all-reduce (exposed communication)."""
    import monodepth2_jl_b200 as M
    from monodepth2_jl_b200 import dist as D
    from monodepth2_jl_b200 import synthetic as SY
    torch.backends.cudnn.allow_tf32 = bool(args.tf32)
    torch.backends.cuda.matmul.allow_tf32 = bool(args.tf32)
    torch.backends.cudnn.benchmark = True
    xs = [SY.synthetic_batch(NB, CH, H_, W_, seed=1000 + 17 * rank + k)[0].to(dev) for k in range(4)]
    steps, warm = args.train_steps, 8
    stream = torch.cuda.current_stream(dev)
    res = {}
    modes = [True] + ([None, False] if world > 1 else [])
    for overlap in modes:
        trainer, model, cache, hp = M.make_training_setup(W_, H_, dev, channels=CH, batch_size=NB * world, automasking=AM, seed=7, overlap=overlap)
        for k in range(warm):
            trainer.step(xs[k % 4])
        barrier()
        ctx = M.Context.get(dev)
        l0 = ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for k in range(steps):
            loss, _ = trainer.step(xs[k % 4])
        e1.record(stream)
        barrier()
        ms = D.max_over_ranks(e0.elapsed_time(e1), device=dev) / steps
        res[overlap] = dict(ms=ms, launches=(ctx.launches - l0) // steps, loss=float(loss), buckets=len(trainer.flat.buckets),
                            params=trainer.flat.total, calls=trainer.flat.calls)
        del trainer, model
        torch.cuda.empty_cache()
    main = res[True]
    out = {"metric": f"train frames/s @{W_}x{H_} R18 stand-in: model fwd + fused view-synthesis loss + bwd + gradient all-reduce + ADAM",
           "value": round(NB * world / (main["ms"] * 1e-3), 1), "unit": "frames/s", "ms_per_step": round(main["ms"], 4), "steps": steps, "warmup": warm,
           "batch_per_gpu": NB, "model": "ResNet-18 encoder + depth decoder (4 scales) + pose decoder, reference architecture, torch.nn / cuDNN "
           "(host framework layers, not this library), fp32" + (" (TF32 convolutions)" if args.tf32 else " (TF32 off)"),
           "parameters": main["params"], "allreduce_bytes_per_step": 4 * main["params"] if world > 1 else 0,
           "allreduce": "NCCL SUM over %d buckets, started from autograd hooks during backward; mean folded into the ADAM launch" % main["buckets"] if world > 1 else "none (1 GPU)",
           "md2_launches": int(main["launches"]), "final_loss": main["loss"]}
    if world > 1:
        out["ms_per_step_without_allreduce"] = round(res[None]["ms"], 4)
        out["ms_per_step_blocking_allreduce"] = round(res[False]["ms"], 4)
        out["exposed_allreduce_us"] = round(1e3 * (main["ms"] - res[None]["ms"]), 1)
        out["exposed_allreduce_us_blocking"] = round(1e3 * (res[False]["ms"] - res[None]["ms"]), 1)
    return out


def run_config1(args):
    """BASELINE.json configs[0]: the triplet optimiser `slow_depth` (src/simple_depth.jl:1-62): 500 ADAM(3e-4) iterations
    over a 416x128 disparity map + 2 poses on one RGB triplet.  Ours: md2_slow_depth, the whole loop on the device (one
    CUDA-graph launch of { prep, march, finish, adam } per iteration).  Reference arm: the oracle's loop on the host cores."""
    from oracle import torch_oracle as O
    W, H, C = 416, 128, 3
    x = O.synthetic_batch(1, C, H, W, seed=42)[0]
    K, invK = O.make_K(W, H)
    iters = 500
    metric = "slow_depth iterations/s @416x128 triplet (disparity map + so3 + translation, ADAM 3e-4)"
    workload = "configs[0]: simple_depth triplet optimisation, 416x128, N=1, C=3, S=2, 1 scale, 500 iterations"
    if args.impl == "reference":
        torch.set_num_threads(os.cpu_count() or 1)
        n = max(3, min(args.steps, 40))
        O.slow_depth(x, K, invK, iters=2)
        t0 = time.time()
        hist = O.slow_depth(x, K, invK, iters=n)[3]
        dt = (time.time() - t0) / n
        cb = {"value": round(1.0 / dt, 3), "unit": "iterations/s", "cores": os.cpu_count(), "kind": "port",
              "sample": f"{n} of the 500 iterations of the same triplet through the PyTorch-CPU restatement (fp32, all host threads)"}
        print(json.dumps({"impl": "reference", "metric": metric, "value": cb["value"], "unit": "iterations/s", "n_gpus": 1, "steps": n, "warmup": 2,
                          "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic triplet", "config": {"workload": workload}, "cpu_baseline": cb,
                          "e2e": {"value": cb["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
                          "loss_first_last": [hist[0], hist[-1]]}), flush=True)
        return
    import monodepth2_jl_b200 as M
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    xg, Kg, iKg = x.to(dev), K.to(dev), invK.to(dev)
    ctx = M.Context.get(dev)
    M.slow_depth(xg, Kg, iKg, iters=20)                      # warm-up: sizes the workspaces, captures the graph
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(dev.index or 0)
    sampler.sample(); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(1, min(args.steps, 20))
    l0 = ctx.launches
    st = torch.cuda.current_stream(dev)
    e0.record(st)
    for _ in range(reps):
        disp, poses, hist = M.slow_depth(xg, Kg, iKg, iters=iters)
    e1.record(st)
    torch.cuda.synchronize(dev)
    sampler.sample(); sampler.stop_flag = True
    ms = e0.elapsed_time(e1) / (reps * iters)
    # end to end: triplet from pinned host memory, 500 iterations, disparity + poses + loss history back to the host
    hx = x.pin_memory()
    h_out = [torch.empty(1, 1, H, W).pin_memory(), torch.empty(iters).pin_memory()]
    t0 = time.perf_counter()
    for _ in range(reps):
        xd = hx.to(dev, non_blocking=True)
        disp, poses, hist = M.slow_depth(xd, Kg, iKg, iters=iters)
        h_out[0].copy_(disp, non_blocking=True); h_out[1].copy_(hist, non_blocking=True)
        pr = [(p.rvec.cpu(), p.tvec.cpu()) for p in poses]
    e_ms = (time.perf_counter() - t0) * 1e3 / (reps * iters)
    abytes, per_unit = algorithmic_bytes(W, H, 1, C, 2, 1, g=0)
    peak, peak_src = peaks()
    out = {"metric": metric, "value": round(1e3 / ms, 1), "unit": "iterations/s", "n_gpus": 1, "steps": reps * iters, "warmup": 20,
           "ms_per_step": round(ms, 5), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic triplet",
           "config": {"workload": workload, "l2_policy": "the triplet IS L2-resident by construction (one 416x128 triplet optimised in place): latency-bound, reported as such",
                      "api": "md2_slow_depth (C ABI) via monodepth2_jl_b200.slow_depth"},
           "gpu_launches": int(ctx.launches - l0), "clocks": sampler.summary(),
           "e2e": {"value": round(1e3 / e_ms, 1), "unit": "iterations/s", "h2d_bytes_per_step": int(4 * x.numel() / iters), "d2h_bytes_per_step": int(4 * (H * W + iters + 12) / iters),
                   "note": "per 500-iteration solve: the triplet travels from pinned host memory once, disparity map, poses and loss history travel back once"},
           "roofline": {"bound": "hbm", "kernel": "march2_kernel<C=3,S=2,AM=0> inside the captured iteration", "achieved": round(abytes / (ms * 1e-3) / 1e9, 1), "peak": peak,
                        "unit": "GB/s", "frac": round(abytes / (ms * 1e-3) / 1e9 / peak, 4), "traffic": None, "algorithmic_bytes_per_launch": abytes, "bytes_per_unit": per_unit,
                        "note": "whole iteration (4 launches) timed, not the kernel alone: 53 k units per launch cannot fill 148 SMs; latency-bound", "peak_source": peak_src},
           "loss_first_last": [float(hist[0]), float(hist[-1])]}
    if not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        O.slow_depth(x, K, invK, iters=2)
        t0 = time.time()
        O.slow_depth(x, K, invK, iters=20)
        dt = (time.time() - t0) / 20
        out["cpu_baseline"] = {"value": round(1.0 / dt, 3), "unit": "iterations/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "20 of the 500 iterations of the same triplet through the PyTorch-CPU restatement (fp32, all host threads)"}
    print(json.dumps(out), flush=True)


def cpu_step(base, K, invK):
    """one step of the reference's CPU path as restated by the oracle (fp32, autograd = Zygote)"""
    from oracle import torch_oracle as O
    x, disps, rv, tv = base
    x = x.clone().requires_grad_(True)   # Zygote also forms the image cotangent inside grid_sample's pullback
    dd = [d.clone().requires_grad_(True) for d in disps]
    rr = [r.clone().requires_grad_(True) for r in rv]
    tt = [t.clone().requires_grad_(True) for t in tv]
    auto = O.automasking_loss(O.SSIM(), x.detach(), x.detach()[:, 1], (0, 2)) if AM else None   # src/Monodepth.jl:159-164
    loss = O.view_synthesis_loss(x, dd, rr, tt, K, invK, automasking=AM, auto_loss=auto)
    loss.backward()
    return loss.item()


def cpu_baseline(base, budget_s=15.0, steps=None, warmup=1, one_thread=True):
    from oracle import torch_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    K, invK = O.make_K(W_, H_)
    for _ in range(warmup):
        cpu_step(base, K, invK)
    times = []
    t_start = time.time()
    while (steps is None and time.time() - t_start < budget_s and len(times) < 50) or (steps is not None and len(times) < steps):
        t0 = time.time()
        cpu_step(base, K, invK)
        times.append(time.time() - t0)
    mean = sum(times) / len(times)
    one = None
    if one_thread:   # the same step on ONE host thread (BASELINE.md section 4)
        torch.set_num_threads(1)
        cpu_step(base, K, invK)
        t0 = time.time()
        cpu_step(base, K, invK)
        one = time.time() - t0
        torch.set_num_threads(cores)
    c_one = None
    if one_thread:   # the scalar C restatement (oracle/c_oracle.c: float64, hand-derived reverse pass), one thread
        try:
            from oracle import c_oracle as CO
            auto = O.automasking_loss(O.SSIM(), base[0], base[0][:, 1], (0, 2)) if AM else None
            t0 = time.time()
            CO.view_synthesis_loss(base[0], base[1], base[2], base[3], K, invK, auto_loss=auto)
            c_one = time.time() - t0
        except Exception as e:   # (no C compiler on the box and no prebuilt library: the figure is optional)
            print(f"c_oracle unavailable: {e}", file=sys.stderr)
    return {"value": round(NB / mean, 3), "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"{len(times)} steps of the same workload (batch {NB}, {W_}x{H_}, 4 scales, fwd+bwd) through the "
                      f"PyTorch-CPU restatement of the reference (Julia is not installed), fp32, {cores} threads; "
                      f"best {NB / min(times):.3f} frames/s", "ms_per_step": round(mean * 1e3, 2),
            "value_1_thread": round(NB / one, 3) if one else None,
            "value_c_oracle_f64_1_thread": round(NB / c_one, 3) if c_one else None}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    from oracle import torch_oracle as O
    base = O.synthetic_batch(NB, CH, H_, W_, seed=42)
    cb = cpu_baseline(base, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 3)))
    out = {
        "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (same seeded batch as the GPU arm)",
        "config": {"workload": WORKLOAD, "note": "reference CPU path timed on rank 0's host cores only; each step is one "
                   "batch of 8 triplets; the reference itself is single-process"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-groups", type=int, default=1, help="image groups inside one synchronous host call (1: the pinned slabs travel as one copy each way)")
    ap.add_argument("--e2e-lanes", type=int, default=3, help="steps in flight in the multi-buffered end-to-end measurement (2 or 3)")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the process to the GPU-local CPUs")
    ap.add_argument("--config", type=int, default=2, choices=[1] + sorted(CONFIGS),
                    help="BASELINE.json configuration (1-based): 2 (default, the metric's), 3, 4; 1 = the slow_depth triplet optimiser")
    ap.add_argument("--train-step", action="store_true", help="make the full data-parallel training step (row F1) the main line")
    ap.add_argument("--no-train-step", action="store_true", help="skip the training-step section")
    ap.add_argument("--train-steps", type=int, default=30, help="timed steps of the training-step section")
    ap.add_argument("--tf32", action="store_true", help="allow TF32 in the stand-in model's convolutions (default: strict fp32)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the loss and gradients of the last timed "
                    "step as float32 DIR/<name>.npy (CUDA arm, configs 2-4)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config == 1):
        ap.error("--dump-outputs writes the outputs of the CUDA view-synthesis loss path (--impl ours, --config 2, 3 or 4)")
    if args.config == 1:
        if int(os.environ.get("RANK", "0")) == 0:
            run_config1(args)
        return
    set_config(args.config)
    if args.impl == "reference":
        if args.steps > 40:
            args.steps = 40   # bounded sample: the CPU arm takes ~1 s per step
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
