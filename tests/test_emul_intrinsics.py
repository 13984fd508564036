"""The intrinsics gradients of the fused path on the CPU: the marching-kernel source (run by tests/emul, here through
tests/emul/md2_emul_intrinsics.cpp) accumulates the per-(source, image) sums G, h; the pose finalisation forms each pair's
contribution to dL/dK and dL/dinvK and the finish kernel's fixed-order reduction sums them.  Compared with the C oracle
evaluated with the kernel's own decisions forced, on small odd shapes with a distinct camera per image, at the bars of
test_emul_forced.py."""
import ctypes as C
import os
import subprocess
import tempfile

import pytest
import torch

from intrinsics_oracle import c_vsl
from monodepth2_jl_b200 import _lib as L
from oracle import torch_oracle as O
from test_oracle_intrinsics import cameras, per_matrix_err
from util import GRAD_RTOL, LOSS_RTOL, rel_max


EMUL = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emul")
CSRC = os.path.join(os.path.dirname(EMUL), "..", "monodepth2.jl_b200", "csrc")


def build():
    """compiled into a per-user temporary directory (the tree may be read-only)"""
    out = os.path.join(tempfile.gettempdir(), f"md2_test_{os.getuid()}")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libmd2_emul_intrinsics.so")
    deps = [os.path.join(EMUL, f) for f in ("md2_emul_intrinsics.cpp", "md2_emul.cpp", "warp_emu.h")] + \
        [os.path.join(CSRC, f) for f in ("md2_fused.cuh", "md2_march.cuh", "md2_march2.cuh", "md2_math.cuh")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        tmp = so + f".{os.getpid()}"
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", tmp,
                        os.path.join(EMUL, "md2_emul_intrinsics.cpp")], check=True)
        os.replace(tmp, so)
    return so


def emul(x, disps, rv, tv, K, invK, auto, R=12):
    lib = C.CDLL(build())
    lib.md2_emul_march2_intrinsics.argtypes = [C.POINTER(L.VslDesc), C.c_int, C.c_float, C.c_int]
    N, F, Cc, H, W = x.shape
    per_image = K.dim() == 3
    cm = lambda m: m.transpose(-1, -2).contiguous()
    Kc, iKc = cm(K), cm(invK)
    out = dict(loss=torch.zeros(1), gdisp=[torch.zeros_like(d) for d in disps], grvec=[torch.zeros_like(r) for r in rv],
               gtvec=[torch.zeros_like(t) for t in tv], gK=torch.zeros_like(Kc), giK=torch.zeros_like(iKc),
               choices=torch.zeros(len(disps), N, H, W, 3, dtype=torch.int32))
    desc = L.make_vsl_desc(
        target=x[:, 1], target_stride=x.stride(0), sources=[x[:, 0], x[:, 2]], source_strides=[x.stride(0)] * 2,
        disparities=disps, K_cm=Kc, invK_cm=iKc, per_image_K=per_image, grad_K=out["gK"], grad_invK=out["giK"],
        rot=rv, trans=tv, pose_mode=1, invert=[True, False], automask=auto,
        smooth_weight=[1e-3 * s for s in (0.125, 0.25, 0.5, 1.0)[:len(disps)]], loss_scale=1.0 / len(disps),
        loss=out["loss"], grad_disparity=out["gdisp"], grad_rot=out["grvec"], grad_trans=out["gtvec"],
        debug_choices=out["choices"], shape=(N, Cc, H, W))
    assert lib.md2_emul_march2_intrinsics(C.byref(desc), 2, 1.0, R) == 0
    out["gK"] = out["gK"].reshape(-1, 3, 3).transpose(1, 2).reshape(K.shape)
    out["giK"] = out["giK"].reshape(-1, 3, 3).transpose(1, 2).reshape(invK.shape)
    return out


@pytest.mark.parametrize("N,C,H,W,am,per_image", [(3, 1, 17, 33, True, True), (2, 3, 30, 37, False, True),
                                                  (2, 1, 21, 29, False, False)])
def test_emulated_kernel_against_forced_c_oracle(N, C, H, W, am, per_image):
    x, disps, rv, tv = O.synthetic_batch(N, C, H, W, seed=N + W)
    K, invK = cameras(N, W, H, seed=H) if per_image else O.make_K(W, H, dtype=torch.float64)
    K, invK = K.float(), invK.float()
    auto = O.automasking_loss(O.SSIM(), x.double(), x.double()[:, 1], (0, 2)).float().contiguous() if am else None
    out = emul(x.contiguous(), [d.contiguous() for d in disps], [r.contiguous() for r in rv], [t.contiguous() for t in tv], K, invK, auto)
    ref = c_vsl(x, disps, rv, tv, K, invK, auto=auto, choices=out["choices"])
    tag = f"{N},{C},{H},{W},{am},{per_image}"
    assert abs(out["loss"].item() - ref["loss"]) <= LOSS_RTOL * abs(ref["loss"]), tag
    assert per_matrix_err(out["gK"].double(), ref["gK"]) <= GRAD_RTOL, (tag, per_matrix_err(out["gK"].double(), ref["gK"]))
    assert per_matrix_err(out["giK"].double(), ref["ginvK"]) <= GRAD_RTOL, (tag, per_matrix_err(out["giK"].double(), ref["ginvK"]))
    for i, (a, b) in enumerate(zip(out["gdisp"], ref["gdisp"])):
        assert rel_max(a, b) <= GRAD_RTOL, (tag, "gdisp", i)
    for name in ("grvec", "gtvec"):
        for s in range(2):
            assert rel_max(out[name][s], ref[name][s]) <= GRAD_RTOL, (tag, name, s)
