"""Per-image camera intrinsics and the gradients with respect to K and invK (md2_vsl_desc.per_image_K / grad_K /
grad_invK) on the GPU: forced-decision parity against both float64 oracles, bitwise invariance of every existing output,
run-to-run stability through the replayed graph, the split and host entry points, md2_warp_bwd, and torch autograd
end to end."""
import ctypes as C

import pytest
import torch

import monodepth2_jl_b200 as M
from monodepth2_jl_b200 import _lib as L
from intrinsics_oracle import c_vsl, torch_loss
from oracle import torch_oracle as O
from util import GRAD_RTOL, LOSS_RTOL, rel_max

pytestmark = pytest.mark.gpu
POSE_RTOL = 1e-4
# A camera per image: each matrix is a sum over ONE image (W H pixels, both sources) of products in which the pixel
# coordinate enters with weight up to W (G = sum cbar (z p)^T is accumulated in float32 with p = (px, py, 1)), and
# dL/dK = G (R invK)^T + h t^T then cancels the principal-point offset (the third column of invK is ~ -(cx, cy) / f).  The
# float32 rounding of G relative to the result is up to ~W/2 times that of a plain sum, and more for an image whose
# gradient is nearly symmetric about the principal point.  Measured on the B200 with the decisions forced, largest over
# the images: 1.5e-4 (416x128x8), 6.2e-4 (640x192x12; the other images 8e-6 .. 4e-4), 2.6e-6 (61x77x3) of the matrix's
# largest element.  A shared camera sums the same terms over all images and meets 1e-4 (measured 2e-6 .. 2e-5).
PER_IMAGE_INTR_RTOL = 1e-3
DEV = torch.device("cuda", 0)


def cameras(N, W, H, seed):
    """distinct per-image K: focal 0.5-0.9 W, principal point within +-10 px of the centre; invK its float64 inverse"""
    g = torch.Generator().manual_seed(seed)
    f = (0.5 + 0.4 * torch.rand(N, 2, generator=g, dtype=torch.float64)) * W
    c = torch.tensor([W / 2.0, H / 2.0], dtype=torch.float64) + (torch.rand(N, 2, generator=g, dtype=torch.float64) - 0.5) * 20
    K = torch.zeros(N, 3, 3, dtype=torch.float64)
    K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2], K[:, 2, 2] = f[:, 0], f[:, 1], c[:, 0], c[:, 1], 1.0
    return K.float(), torch.linalg.inv(K).float()


def cm(K):
    """(3,3) / (N,3,3) natural -> column-major device block"""
    return K.transpose(-1, -2).contiguous().to(DEV)


def nat(g, per_image):
    return g.reshape(-1, 3, 3).transpose(1, 2).cpu() if per_image else g.reshape(3, 3).t().cpu()


def run(x, disps, rv, tv, K, invK, *, automask=None, grad_K=True, choices=False, mode="fwdbwd", pose_mode=1, calls=1):
    """one fused call through the C ABI; K / invK (3,3) shared or (N,3,3) per image (natural convention, CPU)"""
    N, Lf, Cc, H, W = x.shape
    per_image = K.dim() == 3
    xg = x.to(DEV).contiguous()
    dg = [d.to(DEV).contiguous() for d in disps]
    if pose_mode == 1:
        rg, tg = [r.to(DEV).contiguous() for r in rv], [t.to(DEV).contiguous() for t in tv]
    else:
        Ps = [O.composeT(r.double(), t.double(), sid < 1) for r, t, sid in zip(rv, tv, (0, 2))]
        rg = [P[0].float().transpose(1, 2).contiguous().to(DEV) for P in Ps]
        tg = [P[1].float().contiguous().to(DEV) for P in Ps]
    Kc, iKc = cm(K), cm(invK)
    out = dict(loss=torch.zeros((), device=DEV), gdisp=[torch.zeros_like(d) for d in dg], grot=[torch.zeros_like(r) for r in rg],
               gtrans=[torch.zeros_like(t) for t in tg], gx=torch.zeros_like(xg),
               gK=torch.zeros_like(Kc) if grad_K else None, giK=torch.zeros_like(iKc) if grad_K else None,
               choices=torch.zeros(len(disps), N, H, W, 3, dtype=torch.int32, device=DEV) if choices else None,
               saved=torch.zeros(len(disps), N, 4, device=DEV))
    desc = L.make_vsl_desc(
        target=xg[:, 1], target_stride=xg.stride(0), sources=[xg[:, 0], xg[:, 2]], source_strides=[xg.stride(0)] * 2,
        disparities=dg, K_cm=Kc, invK_cm=iKc, per_image_K=per_image, grad_K=out["gK"], grad_invK=out["giK"],
        rot=rg, trans=tg, pose_mode=pose_mode, invert=[pose_mode == 1, False],
        automask=None if automask is None else automask.float().contiguous().to(DEV),
        smooth_weight=[1e-3 * s for s in (0.125, 0.25, 0.5, 1.0)[:len(disps)]], loss_scale=1.0 / len(disps),
        loss=out["loss"], grad_disparity=out["gdisp"], grad_rot=out["grot"], grad_trans=out["gtrans"],
        grad_source=[out["gx"][:, 0], out["gx"][:, 2]], zero_grad_source=True, debug_choices=out["choices"],
        saved=out["saved"], shape=(N, Cc, H, W))
    ctx = L.Context.get(DEV)
    hist = []
    for _ in range(calls):
        if mode == "fwdbwd":
            ctx.call("md2_view_synthesis_loss_fwdbwd", C.byref(desc), 1.0)
        else:
            ctx.call("md2_view_synthesis_loss_fwd", C.byref(desc))
            ctx.call("md2_view_synthesis_loss_bwd", C.byref(desc), 1.0)
        torch.cuda.synchronize()
        hist.append({k: (v.clone().cpu() if torch.is_tensor(v) else [t.clone().cpu() for t in v]) for k, v in out.items()
                     if v is not None and k != "saved"})
    return hist if calls > 1 else hist[0]


def check_intr(a, b, tag, per_image):
    """every element of each (3,3) matrix within GRAD_RTOL (per image: PER_IMAGE_INTR_RTOL) of that matrix's largest
    element"""
    a, b = a.reshape(-1, 3, 3).double(), b.reshape(-1, 3, 3).double()
    tol = PER_IMAGE_INTR_RTOL if per_image else GRAD_RTOL
    errs = [rel_max(a[m], b[m]) for m in range(a.shape[0])]
    print(f"[intrinsics] {tag}: max error {max(errs):.2e} of the matrix's largest element (bar {tol:.0e})")
    assert max(errs) <= tol, (tag, errs)


CONFIGS = [
    pytest.param(8, 1, 128, 416, False, id="c2-416x128x8-C1"),
    pytest.param(12, 3, 192, 640, True, id="c3-640x192x12-C3-automask"),
    pytest.param(3, 1, 77, 61, True, id="odd-61x77x3-C1-automask"),
]


@pytest.mark.parametrize("per_image", [False, True], ids=["shared", "per-image"])
@pytest.mark.parametrize("N,C,H,W,am", CONFIGS)
def test_forced_parity_both_oracles(N, C, H, W, am, per_image):
    x, disps, rv, tv = O.synthetic_batch(N, C, H, W, seed=42)
    K, invK = cameras(N, W, H, seed=N + W) if per_image else O.make_K(W, H)
    auto = M.automasking_loss(M.SSIM(), x.to(DEV), x.to(DEV)[:, 1], (0, 2)).cpu() if am else None
    out = run(x, disps, rv, tv, K, invK, automask=auto, choices=True)
    ch = out["choices"]
    # torch oracle: autograd through K and invK as independent leaves
    Kd, iKd = K.double().requires_grad_(True), invK.double().requires_grad_(True)
    loss = torch_loss(x.double(), [d.double() for d in disps], [r.double() for r in rv], [t.double() for t in tv],
                      Kd, iKd, choices=ch, auto=None if auto is None else auto.double())
    gK, giK = torch.autograd.grad(loss, (Kd, iKd))
    # C oracle: hand-derived reverse pass
    co = c_vsl(x, disps, rv, tv, K, invK, auto=auto, choices=ch)
    tag = f"{N},{C},{H},{W},{am},{per_image}"
    for ref_loss, ref_K, ref_iK in ((loss.item(), gK, giK), (co["loss"], co["gK"], co["ginvK"])):
        assert abs(out["loss"].item() - ref_loss) <= LOSS_RTOL * abs(ref_loss), (tag, out["loss"].item(), ref_loss)
        check_intr(nat(out["gK"], per_image), ref_K, tag + " K", per_image)
        check_intr(nat(out["giK"], per_image), ref_iK, tag + " invK", per_image)
    for i, (a, b) in enumerate(zip(out["gdisp"], co["gdisp"])):
        assert rel_max(a, b) <= GRAD_RTOL, (tag, "gdisp", i, rel_max(a, b))
    for s in range(2):
        assert rel_max(out["grot"][s], co["grvec"][s]) <= POSE_RTOL, (tag, "grvec", s)
        assert rel_max(out["gtrans"][s], co["gtvec"][s]) <= POSE_RTOL, (tag, "gtvec", s)


def test_grad_K_changes_no_other_output_and_is_stable():
    x, disps, rv, tv = O.synthetic_batch(8, 1, 128, 416, seed=7)
    K, invK = O.make_K(416, 128)
    base = run(x, disps, rv, tv, K, invK, grad_K=False)
    hist = run(x, disps, rv, tv, K, invK, grad_K=True, calls=3)     # calls 2 and 3 replay the captured graph
    for h in hist:
        assert torch.equal(h["loss"], base["loss"])
        for name in ("gdisp", "grot", "gtrans"):
            for a, b in zip(h[name], base[name]):
                assert torch.equal(a, b), name
        assert torch.equal(h["gK"], hist[0]["gK"]) and torch.equal(h["giK"], hist[0]["giK"])
    assert hist[0]["gK"].abs().max() > 0


def test_identical_per_image_copies_equal_shared():
    N = 4
    x, disps, rv, tv = O.synthetic_batch(N, 3, 96, 160, seed=11)
    K, invK = O.make_K(160, 96)
    a = run(x, disps, rv, tv, K, invK)
    b = run(x, disps, rv, tv, K.expand(N, 3, 3), invK.expand(N, 3, 3))
    assert torch.equal(a["loss"], b["loss"])
    for name in ("gdisp", "grot", "gtrans"):
        for u, v in zip(a[name], b[name]):
            assert torch.equal(u, v), name
    assert rel_max(nat(b["gK"], True).sum(0), nat(a["gK"], False)) < 1e-6
    assert rel_max(nat(b["giK"], True).sum(0), nat(a["giK"], False)) < 1e-6


@pytest.mark.parametrize("pose_mode", [0, 1])
def test_split_fwd_bwd_equals_fused(pose_mode):
    N = 3
    x, disps, rv, tv = O.synthetic_batch(N, 1, 64, 96, seed=5)
    K, invK = cameras(N, 96, 64, seed=2)
    a = run(x, disps, rv, tv, K, invK, pose_mode=pose_mode)
    b = run(x, disps, rv, tv, K, invK, pose_mode=pose_mode, mode="split")
    assert torch.equal(a["gK"], b["gK"]) and torch.equal(a["giK"], b["giK"])
    for u, v in zip(a["gdisp"] + a["grot"] + a["gtrans"], b["gdisp"] + b["grot"] + b["gtrans"]):
        assert rel_max(u, v) <= 1e-5      # (the split backward reads the forward's statistics: other summation order)


@pytest.mark.parametrize("per_image", [False, True], ids=["shared", "per-image"])
@pytest.mark.parametrize("groups", [1, 2])
def test_host_entry_point_matches_device(groups, per_image):
    N, Cc, H, W = 4, 3, 96, 128
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, seed=3)
    K, invK = cameras(N, W, H, seed=4) if per_image else O.make_K(W, H)
    dev = run(x, disps, rv, tv, K, invK)
    hl = M.HostViewSynthesisLoss(N, Cc, H, W, [(d.shape[-1], d.shape[-2]) for d in disps], K, invK, groups=groups, grad_K=True)
    loss = hl(x=x, disparities=disps, rvecs=rv, tvecs=tv)
    assert abs(loss - dev["loss"].item()) <= LOSS_RTOL * abs(dev["loss"].item())
    for name, ref in (("K", dev["gK"]), ("invK", dev["giK"])):
        check_intr(hl.grads[name], nat(ref, per_image), name, per_image)
    for a, b in zip(hl.grads["disparities"], dev["gdisp"]):
        assert rel_max(a, b) <= GRAD_RTOL


def test_warp_bwd_grad_K_matches_autograd():
    N, Cc, H, W = 2, 3, 40, 56
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, seed=8, full_res_disp=True)
    K, invK = cameras(N, W, H, seed=9)
    Ps = [O.composeT(r.double(), t.double(), False) for r, t in zip(rv, tv)]
    g = torch.Generator().manual_seed(1)
    gouts = [torch.randn(N, Cc, H, W, generator=g) for _ in range(2)]
    # device: md2_warp_bwd through the C ABI
    xg, dg = x.to(DEV).contiguous(), disps[-1].to(DEV).contiguous()
    rg = [P[0].float().transpose(1, 2).contiguous().to(DEV) for P in Ps]
    tg = [P[1].float().contiguous().to(DEV) for P in Ps]
    gK, giK = torch.zeros(N * 9, device=DEV), torch.zeros(N * 9, device=DEV)
    gd = torch.zeros_like(dg)
    Kc, iKc = cm(K), cm(invK)          # (the descriptor holds raw pointers: keep the tensors alive)
    desc = L.make_vsl_desc(
        target=None, target_stride=0, sources=[xg[:, 0], xg[:, 2]], source_strides=[xg.stride(0)] * 2, disparities=[dg],
        K_cm=Kc, invK_cm=iKc, per_image_K=True, grad_K=gK, grad_invK=giK, rot=rg, trans=tg, pose_mode=0,
        invert=[0, 0], smooth_weight=[0.0], loss_scale=1.0, grad_disparity=[gd], grad_rot=[torch.zeros_like(r) for r in rg],
        grad_trans=[torch.zeros_like(t) for t in tg], shape=(N, Cc, H, W))
    keep = [t.to(DEV).contiguous() for t in gouts]
    arr = (C.c_void_p * 2)(*[t.data_ptr() for t in keep])
    L.Context.get(DEV).call("md2_warp_bwd", C.byref(desc), arr)
    torch.cuda.synchronize()
    # oracle: autograd of warp
    Kd, iKd = K.double().requires_grad_(True), invK.double().requires_grad_(True)
    obj = 0.0
    for n in range(N):   # (the oracle's warp takes one camera: image by image)
        out = O.warp(disps[-1][n:n + 1].double(), x[n:n + 1].double(), [(P[0][n:n + 1], P[1][n:n + 1]) for P in Ps],
                     O.Backproject(W, H), O.Project(W, H), iKd[n], Kd[n], 0.1, 100.0, (0, 2))
        obj = obj + sum((o * go[n:n + 1].double()).sum() for o, go in zip(out, gouts))
    rK, riK = torch.autograd.grad(obj, (Kd, iKd))
    # (un-forced: a sample whose float32 and float64 positions straddle a cell border moves the result a little)
    check_intr(nat(gK, True), rK, "warp K", True)
    check_intr(nat(giK, True), riK, "warp invK", True)


def test_learned_intrinsics_end_to_end():
    N, Cc, H, W = 2, 3, 64, 96
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, seed=13)

    def build(fx, fy, cx, cy):
        z, o = torch.zeros_like(fx), torch.ones_like(fx)
        K = torch.stack([torch.stack([fx, z, cx]), torch.stack([z, fy, cy]), torch.stack([z, z, o])])
        return K, torch.linalg.inv(K)
    vals = [0.6 * W, 0.62 * W, W / 2 + 1.5, H / 2 - 2.0]
    p32 = [torch.tensor(v, device=DEV, requires_grad=True) for v in vals]
    K, invK = build(*p32)
    ch = torch.zeros(len(disps), N, H, W, 3, dtype=torch.int32, device=DEV)
    loss = M.view_synthesis_loss(x.to(DEV), [d.to(DEV) for d in disps], [r.to(DEV) for r in rv], [t.to(DEV) for t in tv], K, invK,
                                 debug_choices=ch)
    loss.backward()
    p64 = [torch.tensor(v, dtype=torch.float64, requires_grad=True) for v in vals]
    K64, invK64 = build(*p64)
    ref = O.view_synthesis_loss_forced(x.double(), [d.double() for d in disps], [r.double() for r in rv], [t.double() for t in tv],
                                       K64, invK64, ch.cpu())
    ref.backward()
    g = torch.stack([p.grad.double().cpu() for p in p32])
    r = torch.stack([p.grad for p in p64])
    # (the four parameter gradients add dL/dK and dL/dinvK d invK / d(fx, fy, cx, cy), which cancel in part: one bar for
    # the camera of one image, as above)
    print(f"[intrinsics] learned (fx, fy, cx, cy): max error {rel_max(g, r):.2e}")
    assert rel_max(g, r) <= PER_IMAGE_INTR_RTOL, (g, r)


def test_slow_depth_rejects_intrinsics_gradients():
    N, Cc, H, W = 1, 1, 32, 48
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, seed=1, full_res_disp=True)
    K, invK = O.make_K(W, H)
    xg = x.to(DEV).contiguous()
    d = disps[-1].to(DEV).contiguous()
    r = [t.to(DEV).contiguous() for t in rv]
    t_ = [t.to(DEV).contiguous() for t in tv]
    scratch = dict(loss=torch.zeros((), device=DEV), gd=[torch.zeros_like(d)], gr=[torch.zeros_like(v) for v in r],
                   gt=[torch.zeros_like(v) for v in t_])
    state, clock = torch.zeros(2 * (d.numel() + 12), device=DEV), torch.zeros(2, dtype=torch.int64, device=DEV)
    ctx = L.Context.get(DEV)
    for kw, field in ((dict(grad_K=torch.zeros(9, device=DEV)), "grad_K"), (dict(per_image_K=2), "per_image_K")):
        extra = dict(kw)
        pik = extra.pop("per_image_K", False)
        desc = L.make_vsl_desc(
            target=xg[:, 1], target_stride=xg.stride(0), sources=[xg[:, 0], xg[:, 2]], source_strides=[xg.stride(0)] * 2,
            disparities=[d], K_cm=cm(K), invK_cm=cm(invK), rot=r, trans=t_, pose_mode=1, invert=[True, False],
            smooth_weight=[1.0], loss_scale=1.0, normalize_disparity=False, loss=scratch["loss"], grad_disparity=scratch["gd"],
            grad_rot=scratch["gr"], grad_trans=scratch["gt"], shape=(N, Cc, H, W), **extra)
        if pik:
            desc.per_image_K = pik
        with pytest.raises(L.Md2Error, match=field):
            ctx.call("md2_slow_depth", C.byref(desc), 3, C.c_float(1e-3), C.c_float(0.9), C.c_float(0.999), C.c_float(1e-8),
                     C.c_void_p(state.data_ptr()), C.c_void_p(clock.data_ptr()), None, C.c_int64(0))
