"""The fused hot path behind the reference's loss entry points: `warp` (undefined in the
reference, call at src/simple_depth.jl:30-32) and the tail of `train_loss`
(src/training.jl:29-77), plus the containers that cross the boundary (`Pose`
src/pose_decoder.jl:1-5, `Params` src/Monodepth.jl:32-42, `TrainCache` :44-55).
Frame indices here are 0-based (the Julia binding converts from the reference's 1-based ids).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Sequence, Tuple

import torch

from . import _lib as L
from ._lib import Context, require_cuda
from .ops import SSIM, Backproject, Project, _cm, _f32c, _p, composeT

_F32 = torch.float32


@dataclass
class Pose:
    rvec: torch.Tensor   # (N,3)  so3 rotation   [Julia 3xN]
    tvec: torch.Tensor   # (N,3)  translation    [Julia 3x1xN]


@dataclass
class Params:
    target_size: Tuple[int, int]          # (width, height)
    batch_size: int
    min_depth: float = 0.1
    max_depth: float = 100.0
    disparity_smoothness: float = 1e-3
    frame_ids: List[int] = field(default_factory=lambda: [0, 1, 2])
    automasking: bool = True


@dataclass
class TrainCache:
    ssim: SSIM
    backprojections: Backproject
    projections: Project
    K: torch.Tensor
    invK: torch.Tensor
    target_id: int
    source_ids: Sequence[int]
    scales: Sequence[float]

    def __post_init__(self):
        # column-major copies handed to the C ABI, made once -- for a constant shared camera only: intrinsics that are
        # learned (requires_grad) or given per image go through view_synthesis_loss's differentiable route at every call
        fixed = not (self.K.requires_grad or self.invK.requires_grad) and self.K.numel() == 9 and self.invK.numel() == 9
        self.K_cm = _cm(_f32c(self.K.reshape(3, 3))) if fixed else None
        self.invK_cm = _cm(_f32c(self.invK.reshape(3, 3))) if fixed else None


def _frame_ptr_view(x, idx):
    return x[:, idx]


def _intrinsics(K, invK):
    """K, invK of shape (3,3), (1,3,3) or (M,3,3) (natural maths convention) -> (K, invK) as (M,3,3) views, per_image"""
    Kb, iKb = K.reshape(-1, 3, 3), invK.reshape(-1, 3, 3)
    M = max(Kb.shape[0], iKb.shape[0])
    if Kb.shape[0] not in (1, M) or iKb.shape[0] not in (1, M):
        raise ValueError(f"K {tuple(K.shape)} and invK {tuple(invK.shape)}: expected (3,3), (1,3,3) or (N,3,3)")
    return Kb.expand(M, 3, 3), iKb.expand(M, 3, 3), M > 1


def _intrinsics_cm(Kb, per_image):
    """(M,3,3) natural -> the C ABI's column-major block: one (3,3) for a shared camera, (3,3,M) per image"""
    return _cm(_f32c(Kb.detach() if per_image else Kb.detach()[0]))


class _ViewSynthesisLoss(torch.autograd.Function):
    """loss, d loss/d(disparities, rvecs, tvecs[, x]) through the fused CUDA kernels.  When any
    input needs a gradient the value and the gradient are produced by ONE fused pass
    (md2_view_synthesis_loss_fwdbwd, seed 1) and the pullback only scales them."""

    @staticmethod
    def forward(ctx, cfg, x, *tensors):
        Lc, S = cfg["L"], cfg["S"]
        intr = cfg["grad_K"]                 # K, invK are the last two tensor inputs: gradients wanted
        K_cm, invK_cm = cfg["K_cm"], cfg["invK_cm"]
        if intr:
            K_cm, invK_cm = (_intrinsics_cm(t, cfg["per_image_K"]) for t in tensors[-2:])
        disps = [_f32c(t) for t in tensors[:Lc]]
        rot = [_f32c(t) for t in tensors[Lc:Lc + S]]
        trans = [_f32c(t) for t in tensors[Lc + S:Lc + 2 * S]]
        x = _f32c(x)
        require_cuda(x, *disps, *rot, *trans)
        N, Lf, Cc, H, W = x.shape
        c = Context.get(x.device)
        if cfg["per_image_K"] and K_cm.numel() != 9 * N:
            raise ValueError(f"per-image K / invK: expected {N} matrices, got {K_cm.numel() // 9}")
        need = [ctx.needs_input_grad[2 + i] for i in range(len(tensors))]
        need_x = ctx.needs_input_grad[1] and cfg.get("grad_x", True)
        any_grad = any(need) or need_x
        dev = x.device
        loss = torch.empty((), device=dev, dtype=_F32)
        gd = [torch.empty_like(d) for d in disps] if any_grad else None
        gr = [torch.empty_like(r) for r in rot] if any_grad else None
        gt = [torch.empty_like(t) for t in trans] if any_grad else None
        gx = torch.zeros_like(x) if need_x else None
        gK = torch.empty_like(K_cm) if intr and need[-2] else None
        giK = torch.empty_like(invK_cm) if intr and need[-1] else None
        viz_w = viz_l = None
        if cfg.get("viz"):
            viz_w = [torch.empty(N, Cc, H, W, device=dev, dtype=_F32) for _ in range(S)]
            viz_l = torch.empty(N, 1, H, W, device=dev, dtype=_F32)
        sid, tid = cfg["source_ids"], cfg["target_id"]
        desc = L.make_vsl_desc(
            target=x[:, tid], target_stride=x.stride(0),
            sources=[x[:, i] for i in sid], source_strides=[x.stride(0)] * S,
            disparities=disps, K_cm=K_cm, invK_cm=invK_cm, per_image_K=cfg["per_image_K"], grad_K=gK, grad_invK=giK,
            rot=rot, trans=trans,
            pose_mode=cfg["pose_mode"], invert=cfg["invert"], automask=cfg.get("automask"),
            min_depth=cfg["min_depth"], max_depth=cfg["max_depth"], smooth_weight=cfg["smooth_weight"],
            loss_scale=cfg["loss_scale"], normalize_disparity=cfg["normalize"], loss=loss,
            grad_disparity=gd, grad_rot=gr, grad_trans=gt,
            grad_source=[gx[:, i] for i in sid] if need_x else None,
            viz_warped=viz_w, viz_loss=viz_l, debug_choices=cfg.get("debug_choices") if any_grad else None,
            compute_automask=cfg.get("compute_automask", False), shape=(N, Cc, H, W))
        if any_grad:
            c.call("md2_view_synthesis_loss_fwdbwd", C.byref(desc), 1.0)
            ctx.grads = (gd, gr, gt, gx)
            ctx.intr = None
            if intr:   # column-major (3,3[,M]) -> natural (M,3,3), the shape of the tensor inputs
                nat = lambda g: None if g is None else g.reshape(-1, 3, 3).transpose(1, 2)
                ctx.intr = (nat(gK), nat(giK))
        else:
            c.call("md2_view_synthesis_loss_fwd", C.byref(desc))
            ctx.grads = None
        ctx.pose_mode = cfg["pose_mode"]
        ctx.viz = (viz_w, viz_l)
        ctx.mark_non_differentiable(*([t for t in (viz_w or [])] + ([viz_l] if viz_l is not None else [])))
        if cfg.get("viz"):
            return (loss, viz_l, *viz_w)
        return loss

    @staticmethod
    def backward(ctx, g, *unused):
        gd, gr, gt, gx = ctx.grads
        scale = lambda t: None if t is None else t * g
        intr = [scale(t) for t in ctx.intr] if ctx.intr is not None else []
        return (None, scale(gx), *[scale(t) for t in gd], *[scale(t) for t in gr], *[scale(t) for t in gt], *intr)


def view_synthesis_loss(x, disparities, rot, trans, K, invK, *, target_id=1, source_ids=(0, 2),
                        scales=(0.125, 0.25, 0.5, 1.0), min_depth=0.1, max_depth=100.0,
                        disparity_smoothness=1e-3, auto_loss=None, normalize_disparity=True,
                        smooth_weight=None, loss_scale=None, poses_are_rvec=True, invert=None,
                        return_viz=False, K_cm=None, invK_cm=None, debug_choices=None, compute_automask=False):
    """Everything of train_loss after `model(...)` (src/training.jl:29-77) in fused kernels.

    x (N,L,C,H,W); disparities: list of (N,1,h_i,w_i) at the decoder's native sizes (smaller ones
    are align-corners upsampled like the reference does); rot/trans: per source either
    rvec/tvec (N,3) [poses_are_rvec=True: composeT is fused, invert = source_id < target_id]
    or R (N,3,3)/t (N,3) as returned by composeT.  auto_loss (N,1,H,W) enables automasking.
    Returns the scalar loss (and, if return_viz, the last scale's warp-loss map and warped
    images, which the reference copies out for logging).
    compute_automask=True (with auto_loss=None): the automask map is formed inside the call from the un-warped source
    frames (the pre-pass of src/Monodepth.jl:159-164 folded in; a constant of the loss, as in the reference).
    debug_choices: optional int32 (L,N,H,W,1+S) test hook that receives the kernel's discrete decisions
    (include/md2.h: md2_vsl_desc.debug_choices).
    K, invK: (3,3) or (1,3,3) for one camera, (N,3,3) for a camera per image (a mix broadcasts).  invK is an input of its
    own, as in the reference (it is never derived from K).  When either requires grad, both gradients flow back through
    autograd; K_cm / invK_cm (pre-made column-major copies of a constant shared camera) are then ignored."""
    S, Lc = len(source_ids), len(disparities)
    Kb, iKb, per_image = _intrinsics(K, invK)
    grad_K = torch.is_grad_enabled() and (K.requires_grad or invK.requires_grad)
    if grad_K or per_image:
        K_cm = invK_cm = None
    if invert is None:
        invert = [sid < target_id for sid in source_ids]
    if not poses_are_rvec:
        rot = [_cm(r) for r in rot]
    cfg = dict(L=Lc, S=S, source_ids=list(source_ids), target_id=target_id,
               K_cm=K_cm if K_cm is not None or grad_K else _intrinsics_cm(Kb, per_image),
               invK_cm=invK_cm if invK_cm is not None or grad_K else _intrinsics_cm(iKb, per_image),
               per_image_K=per_image, grad_K=grad_K,
               pose_mode=1 if poses_are_rvec else 0, invert=invert,
               automask=_f32c(auto_loss.detach()) if auto_loss is not None else None,
               min_depth=min_depth, max_depth=max_depth,
               smooth_weight=smooth_weight if smooth_weight is not None else
               [disparity_smoothness * s for s in list(scales)[:Lc]],
               loss_scale=loss_scale if loss_scale is not None else 1.0 / Lc,
               normalize=normalize_disparity, viz=return_viz, debug_choices=debug_choices,
               compute_automask=bool(compute_automask) and auto_loss is None)
    trans = [t.reshape(-1, 3) for t in trans]
    out = _ViewSynthesisLoss.apply(cfg, x, *disparities, *rot, *trans, *((Kb, iKb) if grad_K else ()))
    if return_viz:
        loss, viz_l, *viz_w = out
        return loss, viz_w, viz_l
    return out


class HostViewSynthesisLoss:
    """Value and gradients of the train_loss tail for a caller whose batch lives in HOST memory -- the
    reference's per-step `x = device(x)` ... `cpu(loss)` (src/Monodepth.jl:156-176) folded into one call of
    md2_view_synthesis_loss_fwdbwd_host: image groups are pipelined over copy and compute streams and the
    pipeline is replayed as a CUDA graph.  The object owns pinned input / output buffers of one shape
    (`inputs`, `grads`); fill `inputs` in place (or pass tensors to `__call__`, which copies them in) and
    read `loss` / `grads` after the call.

    Double-buffered form (a data loader one step ahead): `lane_inputs[k]` / `lane_grads[k]`, k = 0, 1, are two
    independent buffer sets; `submit(k)` enqueues a step on lane k and returns at once, `wait(k)` blocks until its
    outputs are in `lane_grads[k]` and returns the loss, so the device-to-host copies of one step overlap the
    host-to-device copies and kernels of the next (md2_view_synthesis_loss_fwdbwd_host_submit / md2_host_wait).

    x (N,3,C,H,W); disparities (N,1,h_i,w_i) per scale; rvecs / tvecs (N,3) per source; K, invK (3,3) for one camera or
    (N,3,3) per image.  grad_K=True: also d loss / d K and d loss / d invK, in grads["K"] / grads["invK"] (the shape of
    K / invK, natural convention; views of pinned column-major buffers)."""

    LANES = 3

    def __init__(self, N, C_, H, W, disp_sizes, K, invK, *, device=None, target_id=1, source_ids=(0, 2),
                 scales=(0.125, 0.25, 0.5, 1.0), min_depth=0.1, max_depth=100.0, disparity_smoothness=1e-3,
                 automask=False, normalize_disparity=True, grad_x=False, groups=2, lanes=1, grad_K=False):
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.ctx = Context.get(dev)
        self.groups, self.S, self.L = int(groups), len(source_ids), len(disp_sizes)
        if not 1 <= lanes <= self.LANES:
            raise ValueError(f"lanes must be in 1 .. {self.LANES}")
        pin = lambda *shape: torch.zeros(*shape, dtype=_F32).pin_memory()

        def slab(shapes, align=64):
            """tensors of the given shapes carved out of ONE pinned allocation (`align`-float alignment): the host entry
            point recognises the stretch and moves it with a single copy at the large-transfer rate of the link"""
            sizes = [int(torch.Size(sh).numel()) for sh in shapes]
            offs, tot = [], 0
            for n in sizes:
                offs.append(tot); tot += (n + align - 1) // align * align
            buf = torch.zeros(tot, dtype=_F32).pin_memory()
            return [buf[o:o + n].view(*sh) for o, n, sh in zip(offs, sizes, shapes)], buf
        Kb, iKb, per_image = _intrinsics(K.detach().cpu(), invK.detach().cpu())
        if per_image and Kb.shape[0] != N:
            raise ValueError(f"per-image K / invK: expected {N} matrices, got {Kb.shape[0]}")
        self._K, self._invK = _intrinsics_cm(Kb, per_image).pin_memory(), _intrinsics_cm(iKb, per_image).pin_memory()
        # (natural-convention view of a pinned column-major output buffer of the shape of K)
        kview = lambda buf: buf.view(-1, 3, 3).transpose(1, 2) if per_image else buf.view(3, 3).t()
        self.lane_inputs, self.lane_grads, self._lane_loss, self._descs = [], [], [], []
        for _ in range(lanes):
            am_in = bool(automask) and automask != "inside"          # a map handed in by the caller ("inside": formed by the call)
            big, in_buf = slab([(N, 3, C_, H, W)] + [(N, 1, h, w) for (w, h) in disp_sizes] + ([(N, 1, H, W)] if am_in else []))
            # (the disparity gradients back to back: the one-copy return route takes only a stretch without gaps, and
            # the kernels store these gradients as scalars, so they need no alignment)
            gbig, out_buf = slab([(N, 1, h, w) for (w, h) in disp_sizes], align=1)
            nd = len(disp_sizes)
            inputs = dict(x=big[0], disparities=big[1:1 + nd], rvecs=[pin(N, 3) for _ in source_ids], tvecs=[pin(N, 3) for _ in source_ids],
                          automask=big[1 + nd] if am_in else None, _slab=in_buf)
            grads = dict(disparities=gbig, rvecs=[pin(N, 3) for _ in source_ids],
                         tvecs=[pin(N, 3) for _ in source_ids], x=pin(N, 3, C_, H, W) if grad_x else None, _slab=out_buf)
            gK_cm = pin(self._K.numel()) if grad_K else None
            giK_cm = pin(self._invK.numel()) if grad_K else None
            if grad_K:
                grads.update(K=kview(gK_cm), invK=kview(giK_cm))
            loss = pin(1)
            x, gx = inputs["x"], grads["x"]
            desc = L.make_vsl_desc(
                target=x[:, target_id], target_stride=x.stride(0), sources=[x[:, i] for i in source_ids],
                source_strides=[x.stride(0)] * self.S, disparities=inputs["disparities"], K_cm=self._K, invK_cm=self._invK,
                rot=inputs["rvecs"], trans=inputs["tvecs"], pose_mode=1, invert=[i < target_id for i in source_ids],
                automask=inputs["automask"], compute_automask=(automask == "inside"), min_depth=min_depth, max_depth=max_depth,
                smooth_weight=[disparity_smoothness * s for s in list(scales)[:self.L]], loss_scale=1.0 / self.L,
                normalize_disparity=normalize_disparity, loss=loss, grad_disparity=grads["disparities"],
                grad_rot=grads["rvecs"], grad_trans=grads["tvecs"],
                grad_source=[gx[:, i] for i in source_ids] if grad_x else None, zero_grad_source=True,
                per_image_K=per_image, grad_K=gK_cm, grad_invK=giK_cm, shape=(N, C_, H, W))
            self.lane_inputs.append(inputs); self.lane_grads.append(grads); self._lane_loss.append(loss); self._descs.append(desc)
        self.inputs, self.grads, self._loss, self.desc = self.lane_inputs[0], self.lane_grads[0], self._lane_loss[0], self._descs[0]
        x = self.inputs["x"]
        self.h2d_bytes = 4 * sum(t.numel() for t in [x] + self.inputs["disparities"] + self.inputs["rvecs"] + self.inputs["tvecs"]
                                 + ([self.inputs["automask"]] if self.inputs["automask"] is not None else [])) + 8 * self._K.numel()
        self.d2h_bytes = 4 + 4 * sum(t.numel() for t in self.grads["disparities"] + self.grads["rvecs"] + self.grads["tvecs"]) \
            + (8 * N * C_ * H * W if grad_x else 0)

    def fill(self, lane=0, x=None, disparities=None, rvecs=None, tvecs=None, automask=None):
        """copies the given (CPU) tensors into the pinned inputs of a lane"""
        inputs = self.lane_inputs[lane]
        if x is not None:
            inputs["x"].copy_(x)
        for name, vals in (("disparities", disparities), ("rvecs", rvecs), ("tvecs", tvecs)):
            if vals is not None:
                for dst, src in zip(inputs[name], vals):
                    dst.copy_(src.reshape(dst.shape))
        if automask is not None:
            inputs["automask"].copy_(automask.reshape(inputs["automask"].shape))

    def __call__(self, x=None, disparities=None, rvecs=None, tvecs=None, automask=None):
        """copies any given (CPU) tensors into the pinned inputs, runs one step, returns the loss as a float"""
        self.fill(0, x, disparities, rvecs, tvecs, automask)
        lib = self.ctx.lib
        if lib.md2_view_synthesis_loss_fwdbwd_host(self.ctx.handle, C.byref(self.desc), 1.0, self.groups):
            raise L.Md2Error(lib.md2_last_error().decode())
        return float(self._loss[0])

    def submit(self, lane):
        """enqueue one step on the lane's buffers; returns at once (the lane's inputs must stay untouched until wait)"""
        lib = self.ctx.lib
        if lib.md2_view_synthesis_loss_fwdbwd_host_submit(self.ctx.handle, C.byref(self._descs[lane]), 1.0, self.groups, lane):
            raise L.Md2Error(lib.md2_last_error().decode())

    def wait(self, lane):
        """block until the lane's step is complete; its gradients are in lane_grads[lane]; returns the loss"""
        lib = self.ctx.lib
        if lib.md2_host_wait(self.ctx.handle, lane):
            raise L.Md2Error(lib.md2_last_error().decode())
        return float(self._lane_loss[lane][0])

    @property
    def loss(self):
        return float(self._loss[0])


class _Warp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cfg, disp, x, *poses):
        S = cfg["S"]
        disp, x = _f32c(disp), _f32c(x)
        rot = [_cm(_f32c(r)) for r in poses[:S]]
        trans = [_f32c(t).reshape(-1, 3) for t in poses[S:]]
        require_cuda(disp, x)
        N, Lf, Cc, H, W = x.shape
        outs = [torch.empty(N, Cc, H, W, device=x.device, dtype=_F32) for _ in range(S)]
        desc = L.make_vsl_desc(
            target=None, target_stride=0, sources=[x[:, i] for i in cfg["source_ids"]],
            source_strides=[x.stride(0)] * S, disparities=[disp], K_cm=cfg["K_cm"], invK_cm=cfg["invK_cm"],
            per_image_K=cfg["per_image_K"], rot=rot, trans=trans, pose_mode=0, invert=[0] * S, min_depth=cfg["min_depth"],
            max_depth=cfg["max_depth"], smooth_weight=[0.0], loss_scale=1.0, shape=(N, Cc, H, W))
        arr = (C.c_void_p * S)(*[o.data_ptr() for o in outs])
        Context.get(x.device).call("md2_warp_fwd", C.byref(desc), arr)
        ctx.save_for_backward(disp, x, *rot, *trans)
        ctx.cfg = cfg
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        cfg = ctx.cfg
        S = cfg["S"]
        disp, x, *rest = ctx.saved_tensors
        rot, trans = rest[:S], rest[S:]
        N, Lf, Cc, H, W = x.shape
        gouts = [_f32c(g) if g is not None else torch.zeros(N, Cc, H, W, device=x.device, dtype=_F32) for g in gouts]
        gd = torch.empty_like(disp)
        gr = [torch.empty_like(r) for r in rot]
        gt = [torch.empty_like(t) for t in trans]
        gx = torch.zeros_like(x) if ctx.needs_input_grad[2] else None
        desc = L.make_vsl_desc(
            target=None, target_stride=0, sources=[x[:, i] for i in cfg["source_ids"]],
            source_strides=[x.stride(0)] * S, disparities=[disp], K_cm=cfg["K_cm"], invK_cm=cfg["invK_cm"],
            per_image_K=cfg["per_image_K"], rot=rot, trans=trans, pose_mode=0, invert=[0] * S, min_depth=cfg["min_depth"],
            max_depth=cfg["max_depth"], smooth_weight=[0.0], loss_scale=1.0, grad_disparity=[gd], grad_rot=gr,
            grad_trans=gt, grad_source=[gx[:, i] for i in cfg["source_ids"]] if gx is not None else None,
            shape=(N, Cc, H, W))
        arr = (C.c_void_p * S)(*[g.data_ptr() for g in gouts])
        Context.get(x.device).call("md2_warp_bwd", C.byref(desc), arr)
        return (None, gd, gx, *[r.transpose(1, 2) for r in gr], *gt)


def warp(disp, x, Ps, backprojections, projections, invKs, Ks, *, min_depth, max_depth, source_ids):
    """The `warp` the reference calls but never defines (src/simple_depth.jl:30-32); body as in
    src/training.jl:48-57: disparity -> depth -> backproject -> per (P, sid): project ->
    grid_sample(border).  disp (N,1,H,W) [Julia (1,W,H,1) in slow_depth], x (N,L,C,H,W),
    Ps = [(R (N,3,3), t (N,3)), ...].  Returns the list of warped images (N,C,H,W).
    `backprojections` / `projections` are accepted for signature parity; the fused kernel
    derives the pixel grid itself."""
    S = len(source_ids)
    Kb, iKb, per_image = _intrinsics(Ks, invKs)
    cfg = dict(S=S, source_ids=list(source_ids), K_cm=_intrinsics_cm(Kb, per_image), invK_cm=_intrinsics_cm(iKb, per_image),
               per_image_K=per_image, min_depth=float(min_depth), max_depth=float(max_depth))
    N = x.shape[0]
    disp = disp.reshape(N, 1, x.shape[-2], x.shape[-1])
    Rs = [P[0] for P in Ps]
    ts = [P[1].reshape(-1, 3) for P in Ps]
    return list(_Warp.apply(cfg, disp, x, *Rs, *ts))


class AsyncViz:
    """Device -> host copies of the visualisation outputs (src/training.jl:34-37,71-74: `cpu(disparity)`, `cpu.(warped)`,
    `cpu(warp_loss)`) that do not stall the training stream: the copy runs on a side stream into pinned buffers (one set
    per shape, reused) and `ticket.get()` waits for it -- normally one step later, when the PNGs are written."""

    class Ticket:
        def __init__(self, event, tensors, unpack):
            self._event, self._tensors, self._unpack = event, tensors, unpack

        def ready(self):
            return self._event.query()

        def get(self):
            self._event.synchronize()
            return self._unpack(self._tensors)

    def __init__(self, device):
        self.device = torch.device(device)
        self.stream = torch.cuda.Stream(device=self.device)
        self._pinned = {}

    def _buf(self, key, t):
        b = self._pinned.get(key)
        if b is None or b.shape != t.shape:
            b = self._pinned[key] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
        return b

    def fetch(self, tensors, unpack=lambda ts: ts):
        """start copying the (device) tensors; the producer is the current stream"""
        ready = torch.cuda.Event()
        ready.record(torch.cuda.current_stream(self.device))
        out = []
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(ready)
            for k, t in enumerate(tensors):
                t = t.detach()
                t.record_stream(self.stream)
                out.append(self._buf(k, t).copy_(t, non_blocking=True))
            done = torch.cuda.Event()
            done.record(self.stream)
        return AsyncViz.Ticket(done, out, unpack)


def train_loss(model, x, auto_loss, cache: TrainCache, parameters: Params, do_visualization=False, viz: "AsyncViz | None" = None):
    """Drop-in for src/training.jl:21-78.  `model(x, source_ids, target_id)` returns
    (disparities, poses) exactly like the reference's Model (src/model.jl:8-20); everything
    after it runs in the fused CUDA path.  Returns (loss, vis_disparity, vis_warped, vis_loss): host copies like the
    reference's when do_visualization, else None.  With `viz` (an AsyncViz) the copies run on a side stream and the
    second return value is a ticket whose .get() yields (vis_disparity, vis_warped, vis_loss); the other two are None."""
    disparities, poses = model(x, cache.source_ids, cache.target_id)
    out = view_synthesis_loss(
        x, list(disparities), [p.rvec for p in poses], [p.tvec for p in poses], cache.K, cache.invK,
        target_id=cache.target_id, source_ids=cache.source_ids, scales=cache.scales,
        min_depth=parameters.min_depth, max_depth=parameters.max_depth,
        disparity_smoothness=parameters.disparity_smoothness,
        auto_loss=auto_loss if parameters.automasking else None, return_viz=do_visualization,
        compute_automask=parameters.automasking and auto_loss is None,     # (no map handed in: the call forms it itself)
        K_cm=cache.K_cm, invK_cm=cache.invK_cm)
    if do_visualization:
        loss, vis_warped, vis_loss = out
        S = len(vis_warped)
        fetcher = viz if viz is not None else AsyncViz(x.device)
        ticket = fetcher.fetch([disparities[-1], vis_loss, *vis_warped], unpack=lambda ts: (ts[0], list(ts[2:2 + S]), ts[1]))
        if viz is not None:
            return loss, ticket, None, None
        vd, vw, vl = ticket.get()      # the reference's synchronous cpu(...) (src/training.jl:34-37,71-74)
        return loss, vd, vw, vl
    return out, None, None, None


def simple_depth_loss(x, disp, poses, K, invK, *, target_id=1, source_ids=(0, 2), min_depth=0.1, max_depth=100.0):
    """Objective of the triplet optimiser `slow_depth` (src/simple_depth.jl:25-41):
    mean(prediction_loss(warp(...))) + smooth_loss(disp, target): one scale, un-normalised
    smoothness with weight 1, in ONE fused kernel pass."""
    return view_synthesis_loss(x, [disp], [p.rvec for p in poses], [p.tvec for p in poses], K, invK,
                               target_id=target_id, source_ids=source_ids, min_depth=min_depth,
                               max_depth=max_depth, normalize_disparity=False, smooth_weight=[1.0], loss_scale=1.0)


class Adam:
    """Flux.Optimise.ADAM(eta, (beta1, beta2)) over a fixed list of CUDA float32 parameter tensors, as ONE fused
    multi-tensor kernel launch per step (md2_adam_step; the reference calls `Flux.Optimise.update!(optimizer, theta,
    grads)`, src/Monodepth.jl:165-171, src/simple_depth.jl:43).  The moments and the step counter live in two device
    tensors (`state`, `clock`) that `state_dict()` / `load_state_dict()` save and restore -- the optimiser half of a
    checkpoint (the reference's BSON dump, src/Monodepth.jl:189-192, keeps the model only and restarts ADAM cold)."""

    def __init__(self, params, lr=1e-4, betas=(0.9, 0.999), eps=1e-8):
        self.params = [p for p in params]
        if not 1 <= len(self.params) <= L.ADAM_MAX_TENSORS:
            raise ValueError(f"1 .. {L.ADAM_MAX_TENSORS} tensors per optimiser (flatten the parameters into one buffer)")
        require_cuda(*self.params)
        for p in self.params:
            L._chk(p, "parameter")
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        dev = self.params[0].device
        self.counts = [p.numel() for p in self.params]
        self.state = torch.zeros(2 * sum(self.counts), device=dev, dtype=_F32)
        self.clock = torch.zeros(2, device=dev, dtype=torch.int64)
        self._ctx = Context.get(dev)
        n = len(self.params)
        self._p = (C.c_void_p * n)(*[p.data_ptr() for p in self.params])
        self._n = (C.c_int64 * n)(*self.counts)

    def step(self, grads=None, grad_scale=1.0):
        """one update; grads default to `p.grad` of every parameter"""
        grads = [p.grad for p in self.params] if grads is None else list(grads)
        for g, p in zip(grads, self.params):
            if g is None or g.shape != p.shape or not g.is_contiguous() or g.dtype != _F32:
                raise ValueError("every parameter needs a contiguous float32 gradient of its own shape")
        g_arr = (C.c_void_p * len(grads))(*[g.data_ptr() for g in grads])
        self._ctx.call("md2_adam_step", len(self.params), self._p, g_arr, self._n, self.state.data_ptr(), self.clock.data_ptr(),
                       self.lr, self.betas[0], self.betas[1], self.eps, float(grad_scale))

    @property
    def steps(self):
        return int(self.clock[0].item())

    def state_dict(self):
        return dict(state=self.state.detach().cpu(), clock=self.clock.detach().cpu(), lr=self.lr, betas=self.betas, eps=self.eps,
                    counts=list(self.counts))

    def load_state_dict(self, sd):
        if list(sd["counts"]) != list(self.counts):
            raise ValueError("optimiser state belongs to other parameter shapes")
        self.state.copy_(sd["state"]); self.clock.copy_(sd["clock"])
        self.lr, self.betas, self.eps = float(sd["lr"]), tuple(sd["betas"]), float(sd["eps"])


def slow_depth(x, K, invK, *, target_id=1, source_ids=(0, 2), min_depth=0.1, max_depth=100.0, iters=500, lr=3e-4,
               log_step=5, on_log=None, disp=None, poses=None):
    """Drop-in for the reference's triplet optimiser (src/simple_depth.jl:1-62): a full-resolution disparity map
    (initial value 0.5) and one (rvec, tvec) pose per source (initial rvec (0, 0, 0.01), tvec 0) are fitted to one frame
    triplet x (N=1,3,C,H,W) with ADAM(3e-4) on  mean(prediction_loss(warp(...))) + smooth_loss(disp, target).
    The whole loop stays on the device (md2_slow_depth: one CUDA-graph launch per iteration); `on_log(iter, disp, poses)`
    is called every `log_step` iterations and on the first, where the reference writes its PNG / prints the poses
    (src/simple_depth.jl:23,46-60).  Returns (disp (N,1,H,W), [Pose, ...], loss history (iters,) on the device)."""
    x = _f32c(x)
    require_cuda(x)
    N, Lf, Cc, H, W = x.shape
    dev = x.device
    S = len(source_ids)
    disp = torch.full((N, 1, H, W), 0.5, device=dev, dtype=_F32) if disp is None else _f32c(disp).clone()
    if poses is None:
        poses = [Pose(torch.tensor([[0.0, 0.0, 0.01]] * N, device=dev, dtype=_F32), torch.zeros(N, 3, device=dev, dtype=_F32)) for _ in source_ids]
    else:
        poses = [Pose(_f32c(p.rvec).clone(), _f32c(p.tvec).reshape(N, 3).clone()) for p in poses]
    loss = torch.empty((), device=dev, dtype=_F32)
    gd = torch.empty_like(disp)
    gr = [torch.empty_like(p.rvec) for p in poses]
    gt = [torch.empty_like(p.tvec) for p in poses]
    Kc, iKc = _cm(_f32c(K.reshape(3, 3))), _cm(_f32c(invK.reshape(3, 3)))   # (column-major copies; they outlive the calls)
    desc = L.make_vsl_desc(
        target=x[:, target_id], target_stride=x.stride(0), sources=[x[:, i] for i in source_ids], source_strides=[x.stride(0)] * S,
        disparities=[disp], K_cm=Kc, invK_cm=iKc, rot=[p.rvec for p in poses],
        trans=[p.tvec for p in poses], pose_mode=1, invert=[i < target_id for i in source_ids], min_depth=min_depth, max_depth=max_depth,
        smooth_weight=[1.0], loss_scale=1.0, normalize_disparity=False, loss=loss, grad_disparity=[gd], grad_rot=gr, grad_trans=gt,
        shape=(N, Cc, H, W))
    state = torch.zeros(2 * (N * H * W + 6 * N * S), device=dev, dtype=_F32)
    clock = torch.zeros(2, device=dev, dtype=torch.int64)
    history = torch.zeros(max(iters, 1), device=dev, dtype=_F32)
    ctx = Context.get(dev)
    done = 0
    while done < iters:
        # the reference logs on iteration 1 and on every multiple of log_step
        nxt = iters if on_log is None else min(iters, 1 if done == 0 else (done // log_step + 1) * log_step)
        ctx.call("md2_slow_depth", C.byref(desc), nxt - done, float(lr), 0.9, 0.999, 1e-8, state.data_ptr(), clock.data_ptr(),
                 history.data_ptr(), history.numel())
        done = nxt
        if on_log is not None and (done == 1 or done % log_step == 0):
            on_log(done, disp, poses)
    return disp, poses, history[:iters]
