"""Decoder layouts other than the usual one, and the long upsample adjoint, against the float64 oracle.

The fused calls pick their prep kernel from the layout of the disparities: the lean kernel serves the usual decoder
layout (at most 4 scales, the low-resolution ones first, exactly one full-resolution scale, last); every other layout --
any order, several full-resolution scales or none, up to 8 scales -- goes to the generic prep kernel, which writes the
upsampled disparities into scratch and forms the smoothness sums.  Each case runs three calls:
  - value + gradient with the kernel's discrete decisions forced onto the oracle, at the strict bars (check_forced);
  - forward only: the loss within 1e-5 of the value + gradient call's;
  - split forward -> backward through `saved` ((L,N,4) in torch order, (4,N,L) in md2.h's Julia order): equal to the fused
    value + gradient call at the bars of test_fwd_bwd_split_equals_fused_and_is_linear.
The finish kernel forms the upsample adjoint of a low-resolution row in passes of 64 full-resolution rows; a low-res height
of 3 under H = 150 sends up to 148 rows to one low-res row (three passes)."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import monodepth2_jl_b200 as M
from monodepth2_jl_b200 import _lib as L
from oracle import torch_oracle as O
from test_gpu_forced import check_forced
from util import LOSS_RTOL, oracle_vsl_forced, rel_max

pytestmark = pytest.mark.gpu


def dev():
    return torch.device("cuda", 0)


def low_passed(N, sizes, seed):
    """disparities of exact sizes (w, h): low-passed noise through a sigmoid, as O.synthetic_batch makes them"""
    g = torch.Generator().manual_seed(seed)
    out = []
    for w, h in sizes:
        d = torch.randn(N, 1, h, w, generator=g, dtype=torch.float64)
        d = F.avg_pool2d(F.pad(d, (2, 2, 2, 2), mode="replicate"), 5, 1)
        out.append(torch.sigmoid(2.0 * d).float())
    return out


def run_case(x, disps, rv, tv, scales, am):
    d = dev()
    N, _, Cc, H, W = x.shape
    Lc = len(disps)
    K, invK = O.make_K(W, H)
    xg = x.to(d).requires_grad_(True)
    dg = [t.to(d).requires_grad_(True) for t in disps]
    rg = [t.to(d).requires_grad_(True) for t in rv]
    tg = [t.to(d).requires_grad_(True) for t in tv]
    auto = M.automasking_loss(M.SSIM(), xg.detach(), xg.detach()[:, 1], (0, 2)) if am else None
    tag = f"{W}x{H}x{N} C={Cc} am={am} sizes={[tuple(t.shape[-1:-3:-1]) for t in disps]}"

    # 1. value + gradient, decisions forced onto the float64 oracle
    ch = torch.zeros(Lc, N, H, W, 3, dtype=torch.int32, device=d)
    loss = M.view_synthesis_loss(xg, dg, rg, tg, K.to(d), invK.to(d), scales=scales, auto_loss=auto, debug_choices=ch)
    loss.backward()
    out = dict(loss=loss.item(), gdisp=[t.grad.cpu() for t in dg], grvec=[t.grad.cpu() for t in rg],
               gtvec=[t.grad.cpu() for t in tg], gx=xg.grad.cpu())
    ref = oracle_vsl_forced(x, disps, rv, tv, K, invK, ch.cpu(), auto=None if auto is None else auto.cpu().double(),
                            scales=scales)
    check_forced(out, ref, tag)

    # 2. forward only
    with torch.no_grad():
        lf = M.view_synthesis_loss(xg.detach(), [t.detach() for t in dg], [t.detach() for t in rg], [t.detach() for t in tg],
                                   K.to(d), invK.to(d), scales=scales, auto_loss=auto)
    assert abs(lf.item() - out["loss"]) <= LOSS_RTOL * abs(out["loss"]), (tag, "forward only", lf.item(), out["loss"])

    # 3. split forward -> backward through `saved`, against the fused call of the C ABI
    xd = x.to(d)
    disps_d, rv_d, tv_d = [t.to(d) for t in disps], [t.to(d) for t in rv], [t.to(d) for t in tv]
    K_cm, invK_cm = K.t().contiguous().to(d), invK.t().contiguous().to(d)
    ctx = M.Context.get(d)

    def call(mode, up=1.0, saved=None):
        o = dict(loss=torch.zeros((), device=d), gd=[torch.zeros_like(t) for t in disps_d],
                 gr=[torch.zeros_like(t) for t in rv_d], gt=[torch.zeros_like(t) for t in tv_d], gx=torch.zeros_like(xd),
                 saved=saved if saved is not None else torch.zeros(Lc, N, 4, device=d))
        desc = L.make_vsl_desc(target=xd[:, 1], target_stride=xd.stride(0), sources=[xd[:, 0], xd[:, 2]],
                               source_strides=[xd.stride(0)] * 2, disparities=disps_d, K_cm=K_cm, invK_cm=invK_cm,
                               rot=rv_d, trans=tv_d, pose_mode=1, invert=[1, 0], automask=auto,
                               smooth_weight=[1e-3 * s for s in scales], loss_scale=1.0 / Lc, loss=o["loss"],
                               grad_disparity=o["gd"], grad_rot=o["gr"], grad_trans=o["gt"],
                               grad_source=[o["gx"][:, 0], o["gx"][:, 2]], saved=o["saved"], shape=(N, Cc, H, W))
        if mode == "fwd":
            ctx.call("md2_view_synthesis_loss_fwd", C.byref(desc))
        elif mode == "bwd":
            ctx.call("md2_view_synthesis_loss_bwd", C.byref(desc), up)
        else:
            ctx.call("md2_view_synthesis_loss_fwdbwd", C.byref(desc), up)
        torch.cuda.synchronize()
        return o

    fused = call("fwdbwd")
    fwd = call("fwd")
    bwd = call("bwd", 1.0, fwd["saved"])
    assert abs(fused["loss"].item() - out["loss"]) <= LOSS_RTOL * abs(out["loss"]), (tag, "C ABI fused", fused["loss"].item())
    assert abs(fwd["loss"].item() - fused["loss"].item()) <= 2e-6 * abs(fused["loss"].item()), (tag, "split loss")
    for name in ("gd", "gr", "gt"):
        for i, (a, b) in enumerate(zip(bwd[name], fused[name])):
            assert rel_max(a, b) < 2e-5, (tag, "split", name, i, rel_max(a, b))
    assert rel_max(bwd["gx"], fused["gx"]) < 2e-5, (tag, "split gx", rel_max(bwd["gx"], fused["gx"]))


# (scales, N, C, H, W, automask): the batch of O.synthetic_batch(scales=...), whose sizes are round(side * scale)
SYNTH = [
    pytest.param((1.0, 0.5, 0.25, 0.125), 2, 3, 72, 104, True, id="reversed-C3-am"),
    pytest.param((1.0, 0.5, 0.25, 0.125), 1, 1, 40, 66, False, id="reversed-C1"),
    pytest.param((0.25, 1.0, 0.5, 1.0), 2, 1, 56, 96, False, id="two-full-res-C1"),
    pytest.param((0.25, 1.0, 0.5, 1.0), 1, 3, 45, 77, True, id="two-full-res-C3-am"),
    pytest.param((0.5,), 2, 3, 48, 80, False, id="half-only-C3"),
    pytest.param((0.25, 0.5), 2, 1, 52, 90, True, id="quarter-half-C1-am"),
    pytest.param((1 / 16, 1 / 8, 1 / 4, 1 / 2, 1.0), 2, 3, 96, 160, True, id="five-scales-C3-am"),
    pytest.param((1 / 32, 1 / 16, 1 / 8, 1 / 4, 1 / 2, 1.0, 1 / 2, 1.0), 2, 1, 128, 256, False, id="eight-scales-C1"),
    pytest.param((1 / 32, 1 / 16, 1 / 8, 1 / 4, 1 / 2, 1.0, 1 / 2, 1.0), 1, 3, 128, 256, True, id="eight-scales-C3-am"),
]


@pytest.mark.parametrize("scales,N,Cc,H,W,am", SYNTH)
def test_decoder_layouts(scales, N, Cc, H, W, am):
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, scales=scales, seed=77)
    run_case(x, disps, rv, tv, scales, am)


# (sizes (w, h) per scale, N, C, H, W, automask): disparity sizes given exactly
EXACT = [
    # the half-resolution limit of check_desc: w = (W+1)/2, h = (H+1)/2 -- the 4-row low-res window of the prep kernels
    # is tightest here.  Usual layout (lean prep kernel), then reversed (generic prep kernel)
    pytest.param(((16, 10), (31, 19), (61, 37)), 2, 3, 37, 61, True, id="half-limit-usual-C3-am"),
    pytest.param(((61, 37), (31, 19), (16, 10)), 2, 1, 37, 61, False, id="half-limit-reversed-C1"),
    pytest.param(((31, 19), (61, 37)), 1, 1, 37, 61, True, id="half-limit-usual-C1-am"),
    pytest.param(((61, 37), (31, 19)), 1, 3, 37, 61, False, id="half-limit-reversed-C3"),
    # long adjoint: low-res height 3 under H = 150 (a low-res row receives up to 148 full-resolution rows, three passes
    # of 64); W % 4 == 0 takes the vector phase of the adjoint, W % 4 != 0 the scalar one
    pytest.param(((25, 3), (100, 150)), 2, 1, 150, 100, False, id="long-adjoint-W100-C1"),
    pytest.param(((25, 3), (100, 150)), 1, 3, 150, 100, True, id="long-adjoint-W100-C3-am"),
    pytest.param(((26, 3), (101, 150)), 2, 3, 150, 101, False, id="long-adjoint-W101-C3"),
    pytest.param(((51, 2), (101, 150)), 1, 1, 150, 101, True, id="long-adjoint-W101-h2-C1-am"),
    pytest.param(((101, 150), (25, 3), (50, 75)), 1, 1, 150, 101, False, id="long-adjoint-generic-C1"),
]


@pytest.mark.parametrize("sizes,N,Cc,H,W,am", EXACT)
def test_exact_sizes(sizes, N, Cc, H, W, am):
    x, _, rv, tv = O.synthetic_batch(N, Cc, H, W, scales=(1.0,), seed=91)
    disps = low_passed(N, sizes, seed=92)
    scales = [w / W for w, _ in sizes]
    run_case(x, disps, rv, tv, scales, am)
