"""Stand-alone operators (md2_ops.cu, the drop-in methods of the Julia binding) at the shapes and arguments where their
code paths switch, against the float64 operators of oracle/torch_oracle.py.  Arguments the autograd wrappers of ops.py never
pass (a mask, gmask, argmin = NULL, an image stride other than C*H*W, a non-zero ginput to accumulate into) go through ctypes.
  - project_bwd / warp_bwd sum per-block partials over min(128, ceil(HW / 1024)) blocks: 52 and 128 blocks here;
  - smooth_loss uses min(64, ceil(HW / 2048)) blocks;
  - photometric_min stages interior tiles with bulk copies when C * S >= 4 and W % 4 == 0, through the threads otherwise;
  - grid_sample_bwd merges the scatter of neighbouring lanes that share a cell (zoom-in grid);
  - upsample: non-integer ratios, a one-pixel side, a shrink.
Bars: values 1e-5 and gradients 1e-4 of the array's largest element, except where the existing operator tests of
tests/test_gpu_ops.py allow more (warp: flips of the gather cell, see there)."""
import ctypes as C

import pytest
import torch

import monodepth2_jl_b200 as M
from oracle import torch_oracle as O
from util import rel_max

pytestmark = pytest.mark.gpu
F64 = torch.float64


def dev():
    return torch.device("cuda", 0)


def ctx():
    return M.Context.get(dev())


def pair(t):
    return t.to(dev()).requires_grad_(True), t.double().requires_grad_(True)


def close(a, b, tol, tag=""):
    assert rel_max(a, b) <= tol, (tag, rel_max(a, b))


def ptrs(ts):
    arr = (C.c_void_p * len(ts))()
    for i, t in enumerate(ts):
        arr[i] = None if t is None else t.data_ptr()
    return arr


def p(t):
    return None if t is None else t.data_ptr()


BIG = [pytest.param(128, 416, id="416x128"), pytest.param(320, 1024, id="1024x320")]


# ---------------- project_bwd / warp_bwd: many blocks of per-block partials ----------------
@pytest.mark.parametrize("H,W", BIG)
def test_project_bwd_many_blocks(H, W):
    torch.manual_seed(11)
    N = 2
    K, invK = O.make_K(W, H)
    depth_g, depth_c = pair(torch.rand(N, W * H) * 5 + 1)
    rg, rc = pair(0.05 * torch.randn(N, 3))
    tg, tc = pair(0.05 * torch.randn(N, 3))
    w = torch.randn(N, W * H, 2)
    Rg, tug = M.composeT(rg, tg, True)
    uvg = M.Project(W, H)(M.Backproject(W, H)(depth_g, invK.to(dev())), K.to(dev()), Rg, tug)
    (uvg * w.to(dev())).sum().backward()
    Rc, tuc = O.composeT(rc, tc, True)
    uvc = O.Project(W, H)(O.Backproject(W, H)(depth_c, invK.double()), K.double(), Rc, tuc)
    (uvc * w.double()).sum().backward()
    close(uvg, uvc, 1e-5, "uv")
    close(depth_g.grad, depth_c.grad, 1e-4, "depth")
    close(rg.grad, rc.grad, 1e-4, "rvec")
    close(tg.grad, tc.grad, 1e-4, "tvec")


@pytest.mark.parametrize("H,W", BIG)
def test_warp_bwd_many_blocks(H, W):
    N, Cc = 2, 3
    _, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, scales=(1.0,), seed=4)
    K, invK = O.make_K(W, H)
    d = dev()
    g = torch.Generator().manual_seed(5)
    # smooth frames (no pixel noise) and upstream weights of one sign: a sample that takes the neighbouring cell (its
    # position is within float32 rounding of the border; more of them the larger W) then changes its slope, and with it
    # the pose sums, by little against sums that do not cancel.  The many-block reduction is what is under test here.
    yy, xx = torch.meshgrid(torch.arange(H, dtype=F64), torch.arange(W, dtype=F64), indexing="ij")
    f = lambda: 0.02 + 0.06 * torch.rand((), generator=g, dtype=F64)
    x = torch.stack([torch.stack([torch.stack([0.5 + 0.2 * torch.sin(f() * xx + f() * yy + 6.0 * f()) + 0.1 * torch.cos(f() * xx - f() * yy)
                                               for _ in range(Cc)]) for _ in range(3)]) for _ in range(N)]).float()
    dg, dc = pair(disps[-1])
    rg = [pair(r) for r in rv]
    tg = [pair(t) for t in tv]
    xg, xc = pair(x)
    wts = [1.0 + 0.5 * torch.rand(N, Cc, H, W, generator=g) for _ in range(2)]
    Ps_g = [M.composeT(r[0], t[0], inv) for r, t, inv in zip(rg, tg, (True, False))]
    outs_g = M.warp(dg, xg, Ps_g, M.Backproject(W, H), M.Project(W, H), invK.to(d), K.to(d),
                    min_depth=0.1, max_depth=100.0, source_ids=(0, 2))
    sum(((o * w.to(d)).sum() for o, w in zip(outs_g, wts))).backward()
    Ps_c = [O.composeT(r[1], t[1], inv) for r, t, inv in zip(rg, tg, (True, False))]
    outs_c = O.warp(dc, xc, Ps_c, O.Backproject(W, H), O.Project(W, H), invK.double(), K.double(), 0.1, 100.0, (0, 2))
    sum(((o * w.double()).sum() for o, w in zip(outs_c, wts))).backward()
    # the allowances of test_warp_matches_oracle_and_grads: a sample within float32 rounding of a cell border may take
    # the other cell, which moves its disparity gradient and the pose sums
    for a, b in zip(outs_g, outs_c):
        close(a, b, 2e-5, "warped")
    err = (dg.grad.cpu().double() - dc.grad).abs() / dc.grad.abs().max()
    assert (err <= 1e-4).double().mean().item() >= 0.995, (err <= 1e-4).double().mean().item()
    close(xg.grad, xc.grad, 2e-4, "x")
    for (a, b) in rg + tg:
        close(a.grad, b.grad, 2e-3, "pose")


# ---------------- smooth_loss: many blocks, normalize, image given as a frame of a 5-D tensor ----------------
@pytest.mark.parametrize("frame", [False, True], ids=["image", "frame1"])
@pytest.mark.parametrize("normalize", [False, True], ids=["raw", "normalized"])
@pytest.mark.parametrize("Cc", [1, 3])
@pytest.mark.parametrize("H,W", BIG)
def test_smooth_loss_routes(H, W, Cc, normalize, frame):
    g = torch.Generator().manual_seed(H + Cc)
    N = 2
    disp = torch.rand(N, H, W, generator=g) * 0.9 + 0.1
    x5 = torch.rand(N, 3, Cc, H, W, generator=g)
    img = x5[:, 1] if frame else x5[:, 1].contiguous()
    dev_x5 = x5.to(dev())
    img_d = dev_x5[:, 1] if frame else img.to(dev())
    stride = 3 * Cc * H * W if frame else Cc * H * W
    disp_d = disp.to(dev())
    out = torch.zeros((), device=dev())
    gdisp = torch.empty(N, H, W, device=dev())
    gimg = torch.empty(N, Cc, H, W, device=dev())
    ctx().call("md2_smooth_loss_fwd", p(disp_d), p(img_d), stride, p(out), int(normalize), W, H, Cc, N)
    ctx().call("md2_smooth_loss_bwd", p(disp_d), p(img_d), stride, 1.7, p(gdisp), p(gimg), int(normalize), W, H, Cc, N)
    torch.cuda.synchronize()
    dc = disp.double().requires_grad_(True)
    ic = img.double().requires_grad_(True)
    dn = dc / (dc.mean(dim=(1, 2), keepdim=True) + 1e-7) if normalize else dc
    ref = O.smooth_loss(dn, ic)
    (ref * 1.7).backward()
    assert abs(out.item() - ref.item()) <= 1e-5 * abs(ref.item()), (out.item(), ref.item())
    close(gdisp.cpu(), dc.grad, 1e-4, "gdisp")
    close(gimg.cpu(), ic.grad, 1e-4, "gimage")


# ---------------- photometric_min: mask / gmask / argmin = NULL, copy-engine and thread routes ----------------
PHOTO = [
    # S, C, W, off, mask
    pytest.param(2, 3, 72, 0, True, id="S2-C3-W72-mask"),
    pytest.param(2, 3, 128, 0, False, id="S2-C3-W128"),
    pytest.param(2, 3, 128, 1, True, id="S2-C3-W128-off1-mask"),
    pytest.param(2, 3, 99, 0, False, id="S2-C3-W99"),
    pytest.param(2, 1, 99, 0, True, id="S2-C1-W99-mask"),
    pytest.param(2, 1, 128, 0, False, id="S2-C1-W128"),
    pytest.param(1, 3, 128, 0, True, id="S1-C3-W128-mask"),
    pytest.param(1, 1, 72, 0, True, id="S1-C1-W72-mask"),
    pytest.param(1, 1, 72, 0, False, id="S1-C1-W72-no-argmin"),
    pytest.param(1, 3, 99, 1, False, id="S1-C3-W99-off1-no-argmin"),
    pytest.param(1, 3, 128, 0, False, id="S1-C3-W128-no-argmin"),
]


@pytest.mark.parametrize("S,Cc,W,off,use_mask", PHOTO)
def test_photometric_min_routes(S, Cc, W, off, use_mask):
    N, H = 2, 70
    g = torch.Generator().manual_seed(W + 7 * S + Cc + off)
    buf = torch.rand(N * 3 * Cc * H * W + off, generator=g)
    x = buf[off:].view(N, 3, Cc, H, W)
    xd = buf.to(dev())[off:].view(N, 3, Cc, H, W)
    sids = (0, 2) if S == 2 else (2,)
    mask = (torch.rand(N, 1, H, W, generator=g) * 0.3) if use_mask else None
    mask_d = mask.to(dev()) if use_mask else None
    want_argmin = S > 1 or use_mask
    out = torch.empty(N, 1, H, W, device=dev())
    argmin = torch.full((N, 1, H, W), -7, dtype=torch.int32, device=dev()) if want_argmin else None
    strides = (C.c_int64 * S)(*([xd.stride(0)] * S))
    preds = ptrs([xd[:, s] for s in sids])
    ctx().call("md2_photometric_min_fwd", S, preds, strides, p(xd[:, 1]), xd.stride(0), p(mask_d), 0.85, p(out), p(argmin),
               W, H, Cc, N)
    gout = torch.randn(N, 1, H, W, generator=g)
    gpred = [torch.empty(N, Cc, H, W, device=dev()) for _ in sids]
    gtarget = torch.empty(N, Cc, H, W, device=dev())
    gmask = torch.empty(N, 1, H, W, device=dev()) if use_mask else None
    ctx().call("md2_photometric_min_bwd", S, preds, strides, p(xd[:, 1]), xd.stride(0), p(mask_d), 0.85, p(gout.to(dev())),
               p(argmin), ptrs(gpred), p(gtarget), p(gmask), W, H, Cc, N)
    torch.cuda.synchronize()

    xc = x.double().requires_grad_(True)
    mc = mask.double().requires_grad_(True) if use_mask else None
    pes = [O.photometric_loss(O.SSIM(), xc[:, s], xc[:, 1]) for s in sids]
    stack = torch.cat(([mc] if use_mask else []) + pes, 1)                  # index k: -1 = mask, else source k
    am = argmin.cpu().long() if want_argmin else torch.zeros(N, 1, H, W, dtype=torch.long)
    assert ((am >= (-1 if use_mask else 0)) & (am < S)).all()
    ref = torch.gather(stack, 1, am + (1 if use_mask else 0))                # the oracle with the kernel's arg-min forced
    (ref * gout.double()).sum().backward()
    close(out.cpu(), ref, 1e-5, "out")
    for s, gp in zip(sids, gpred):
        close(gp.cpu(), xc.grad[:, s], 1e-4, f"gpred {s}")
    close(gtarget.cpu(), xc.grad[:, 1], 1e-4, "gtarget")
    if use_mask:
        close(gmask.cpu(), mc.grad, 1e-4, "gmask")
    if stack.shape[1] > 1:
        # the kernel's arg-min is the float64 one (first index wins) wherever the float64 margin exceeds the float32 error
        # radius of the photometric error (r_pe of util.fragile_pixels)
        v = stack.detach()
        top2 = v.topk(2, dim=1, largest=False).values
        clear = (top2[:, 1:2] - top2[:, 0:1]) > 4e-6
        ref_idx = v.argmin(dim=1, keepdim=True) - (1 if use_mask else 0)
        assert clear.double().mean().item() > 0.99
        assert torch.equal(am[clear], ref_idx[clear])


# ---------------- grid_sample_bwd: accumulation into ginput, merged scatter, shared taps, both borders ----------------
def _grid(kind, N, W, H, g):
    if kind == "zoom":        # 8 lanes per cell along x (Wo = 8 (W-1)): neighbouring lanes share taps, the scatter merges
        ix = torch.arange(8 * (W - 1), dtype=F64) / 8 + 1 / 16
        iy = torch.arange(4 * (H - 1), dtype=F64) / 4 + 1 / 8
        gy, gx = torch.meshgrid(iy, ix, indexing="ij")
        gx, gy = gx.expand(N, -1, -1), gy.expand(N, -1, -1)
    elif kind == "constant":  # every lane on the same four taps
        gx = torch.full((N, 24, 40), 5.3, dtype=F64)
        gy = torch.full((N, 24, 40), 3.7, dtype=F64)
    else:                     # beyond both borders, at least 1e-2 of a cell from an integer
        fx = torch.floor(torch.rand(N, 21, 33, generator=g, dtype=F64) * (W + 5)) - 3
        fy = torch.floor(torch.rand(N, 21, 33, generator=g, dtype=F64) * (H + 5)) - 3
        gx = fx + 0.01 + 0.98 * torch.rand(N, 21, 33, generator=g, dtype=F64)
        gy = fy + 0.01 + 0.98 * torch.rand(N, 21, 33, generator=g, dtype=F64)
    return torch.stack([2 * gx / (W - 1) - 1, 2 * gy / (H - 1) - 1], -1).float().contiguous()


@pytest.mark.parametrize("kind", ["zoom", "constant", "beyond"])
@pytest.mark.parametrize("mode", ["zeros", "border"])
@pytest.mark.parametrize("Cc", [1, 3])
def test_grid_sample_bwd_routes(kind, mode, Cc):
    N, H, W = 2, 9, 17                       # W - 1, H - 1 powers of two
    g = torch.Generator().manual_seed(3 * Cc + len(kind))
    inp = torch.rand(N, Cc, H, W, generator=g)
    grid = _grid(kind, N, W, H, g)
    Ho, Wo = grid.shape[1], grid.shape[2]
    gout = torch.randn(N, Cc, Ho, Wo, generator=g)
    init = 0.1 * torch.randn(N, Cc, H, W, generator=g)
    pm = 0 if mode == "zeros" else 1
    inp_d, grid_d = inp.to(dev()), grid.to(dev())
    out = torch.empty(N, Cc, Ho, Wo, device=dev())
    ginput, ggrid = init.to(dev()), torch.empty_like(grid_d)
    ctx().call("md2_grid_sample_fwd", p(inp_d), p(grid_d), p(out), W, H, Cc, N, Wo, Ho, pm)
    ctx().call("md2_grid_sample_bwd", p(inp_d), p(grid_d), p(gout.to(dev())), p(ginput), p(ggrid), W, H, Cc, N, Wo, Ho, pm)
    torch.cuda.synchronize()
    ic, gc = inp.double().requires_grad_(True), grid.double().requires_grad_(True)
    ref = O.grid_sample(ic, gc, padding_mode=mode)
    (ref * gout.double()).sum().backward()
    close(out.cpu(), ref, 1e-5, "out")
    # ACCUMULATED: the result is the starting value plus the gradient
    err = (ginput.cpu().double() - (init.double() + ic.grad)).abs().max() / ic.grad.abs().max()
    assert err.item() <= 1e-5, ("ginput", err.item())
    close(ggrid.cpu(), gc.grad, 1e-4, "ggrid")


# ---------------- upsample: non-integer ratios, one-pixel sides, a shrink ----------------
@pytest.mark.parametrize("w,h,W,H", [(7, 5, 100, 37), (1, 5, 64, 20), (5, 1, 64, 20), (2, 3, 416, 128), (40, 30, 13, 11)])
def test_upsample_routes(w, h, W, H):
    g = torch.Generator().manual_seed(w * 100 + h)
    xg, xc = pair(torch.rand(2, 3, h, w, generator=g))
    wt = torch.randn(2, 3, H, W, generator=g)
    og = M.upsample_bilinear(xg, (W, H))
    (og * wt.to(dev())).sum().backward()
    oc = O.upsample_bilinear(xc, (W, H))
    (oc * wt.double()).sum().backward()
    close(og, oc, 1e-5, "out")
    close(xg.grad, xc.grad, 1e-5, "grad")


# ---------------- ssim: a full-size frame and thin planes ----------------
@pytest.mark.parametrize("shape", [(2, 3, 128, 416), (2, 3, 2, 70), (2, 1, 2, 33), (2, 3, 50, 2), (1, 1, 41, 2)])
def test_ssim_routes(shape):
    g = torch.Generator().manual_seed(sum(shape))
    xg, xc = pair(torch.rand(*shape, generator=g))
    yg, yc = pair(torch.rand(*shape, generator=g))
    wt = torch.randn(*shape, generator=g)
    og = M.SSIM()(xg, yg)
    (og * wt.to(dev())).sum().backward()
    oc = O.SSIM()(xc, yc)
    (oc * wt.double()).sum().backward()
    close(og, oc, 1e-5, "out")
    close(xg.grad, xc.grad, 1e-4, "gx")
    close(yg.grad, yc.grad, 1e-4, "gy")
