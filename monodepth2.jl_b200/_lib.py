"""ctypes binding of libmd2_b200.so (include/md2.h).  There is no CPU fallback: if the shared
library has not been built, or no CUDA device is present, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

MAX_S = 2
MAX_L = 8
HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libmd2_b200.so")

c_float_p = C.POINTER(C.c_float)
c_void = C.c_void_p


class VslDesc(C.Structure):
    """mirror of md2_vsl_desc (include/md2.h)"""
    _fields_ = [
        ("W", C.c_int32), ("H", C.c_int32), ("N", C.c_int32), ("C", C.c_int32), ("S", C.c_int32), ("L", C.c_int32),
        ("target", c_void), ("target_image_stride", C.c_int64),
        ("source", c_void * MAX_S), ("source_image_stride", C.c_int64 * MAX_S),
        ("disparity", c_void * MAX_L),
        ("disp_w", C.c_int32 * MAX_L), ("disp_h", C.c_int32 * MAX_L),
        ("K", c_void), ("invK", c_void),
        ("pose_mode", C.c_int32),
        ("rot", c_void * MAX_S), ("trans", c_void * MAX_S), ("invert", C.c_int32 * MAX_S),
        ("automask", c_void),
        ("min_depth", C.c_float), ("max_depth", C.c_float),
        ("smooth_weight", C.c_float * MAX_L),
        ("loss_scale", C.c_float), ("normalize_disparity", C.c_int32),
        ("loss", c_void),
        ("grad_disparity", c_void * MAX_L),
        ("grad_rot", c_void * MAX_S), ("grad_trans", c_void * MAX_S),
        ("grad_source", c_void * MAX_S),
        ("viz_warped", c_void * MAX_S), ("viz_loss", c_void),
        ("saved", c_void),
        ("zero_grad_source", C.c_int32),
        ("debug_choices", c_void),
        ("compute_automask", C.c_int32),
        ("per_image_K", C.c_int32),
        ("grad_K", c_void), ("grad_invK", c_void),
    ]


def _ptr(t):
    return None if t is None else t.data_ptr()


def _chk(t, name):
    if t is None:
        return
    if t.dtype != torch.float32:
        raise TypeError(f"{name}: expected float32, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: expected a contiguous tensor")


def frame_view(x, idx):
    """(pointer tensor, per-image element stride) of frame `idx` of x (N,L,C,H,W) -- no copy."""
    v = x[:, idx]
    return v, x.stride(0)


def make_vsl_desc(*, target, target_stride, sources, source_strides, disparities, K_cm, invK_cm, rot, trans,
                  pose_mode, invert, automask=None, min_depth=0.1, max_depth=100.0, smooth_weight, loss_scale,
                  normalize_disparity=True, loss=None, grad_disparity=None, grad_rot=None, grad_trans=None,
                  grad_source=None, viz_warped=None, viz_loss=None, saved=None, zero_grad_source=False, debug_choices=None,
                  compute_automask=False, per_image_K=False, grad_K=None, grad_invK=None, shape):
    """shape = (N, C, H, W).  `target`/`sources` are tensors whose data_ptr() is element
    (n=0,c=0,y=0,x=0) of an (N,C,H,W) view with per-image stride *_stride and dense C,H,W.
    per_image_K: K_cm / invK_cm hold N column-major (3,3) matrices (9 N floats) instead of one."""
    N, Cc, H, W = shape
    S, L = len(sources), len(disparities)
    if S > MAX_S or L > MAX_L:
        raise ValueError("too many sources / scales")
    d = VslDesc()
    d.W, d.H, d.N, d.C, d.S, d.L = W, H, N, Cc, S, L
    d.target = _ptr(target)
    d.target_image_stride = target_stride
    for s in range(S):
        d.source[s] = _ptr(sources[s])
        d.source_image_stride[s] = source_strides[s]
        _chk(rot[s], "rot"); _chk(trans[s], "trans")
        d.rot[s] = _ptr(rot[s])
        d.trans[s] = _ptr(trans[s])
        d.invert[s] = int(bool(invert[s]))
        if grad_rot is not None:
            d.grad_rot[s] = _ptr(grad_rot[s])
        if grad_trans is not None:
            d.grad_trans[s] = _ptr(grad_trans[s])
        if grad_source is not None:
            d.grad_source[s] = _ptr(grad_source[s])
        if viz_warped is not None:
            d.viz_warped[s] = _ptr(viz_warped[s])
    for l in range(L):
        _chk(disparities[l], "disparity")
        d.disparity[l] = _ptr(disparities[l])
        d.disp_w[l] = disparities[l].shape[-1]
        d.disp_h[l] = disparities[l].shape[-2]
        d.smooth_weight[l] = float(smooth_weight[l])
        if grad_disparity is not None:
            d.grad_disparity[l] = _ptr(grad_disparity[l])
    _chk(K_cm, "K"); _chk(invK_cm, "invK"); _chk(automask, "automask")
    d.K, d.invK = _ptr(K_cm), _ptr(invK_cm)
    d.pose_mode = pose_mode
    d.automask = _ptr(automask)
    d.min_depth, d.max_depth = float(min_depth), float(max_depth)
    d.loss_scale = float(loss_scale)
    d.normalize_disparity = int(bool(normalize_disparity))
    d.loss = _ptr(loss)
    d.viz_loss = _ptr(viz_loss)
    d.saved = _ptr(saved)
    d.zero_grad_source = int(bool(zero_grad_source))
    d.compute_automask = int(bool(compute_automask))
    nk = 9 * N if per_image_K else 9
    for t, name in ((K_cm, "K"), (invK_cm, "invK"), (grad_K, "grad_K"), (grad_invK, "grad_invK")):
        _chk(t, name)
        if t is not None and t.numel() != nk:
            raise ValueError(f"{name}: expected {nk} floats, got {t.numel()}")
    d.per_image_K = int(bool(per_image_K))
    d.grad_K, d.grad_invK = _ptr(grad_K), _ptr(grad_invK)
    if debug_choices is not None:
        if debug_choices.dtype != torch.int32 or not debug_choices.is_contiguous():
            raise TypeError("debug_choices: expected a contiguous int32 tensor")
        d.debug_choices = debug_choices.data_ptr()
    return d


_I32, _I64, _F = C.c_int32, C.c_int64, C.c_float
_P = c_void   # device pointers travel as void*

_SIGS = {
    "md2_create": [C.c_int, C.POINTER(c_void)],
    "md2_destroy": [c_void],
    "md2_profile_enable": [c_void, _I32],
    "md2_profile_read": [c_void, C.POINTER(C.c_float), C.POINTER(C.c_int64)],
    "md2_profile_read_phases": [c_void, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int64)],
    "md2_disparity_to_depth_fwd": [c_void, _P, _P, _I64, _F, _F, _P],
    "md2_disparity_to_depth_bwd": [c_void, _P, _P, _P, _I64, _F, _F, _P],
    "md2_backproject_fwd": [c_void, _P, _P, _P, _I32, _I32, _I32, _P],
    "md2_backproject_bwd": [c_void, _P, _P, _P, _I32, _I32, _I32, _P],
    "md2_project_fwd": [c_void, _P, _P, _P, _P, _P, _I32, _I32, _I32, _P],
    "md2_project_bwd": [c_void, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _P],
    "md2_so3_exp_map_fwd": [c_void, _P, _P, _I32, _P],
    "md2_so3_exp_map_bwd": [c_void, _P, _P, _P, _I32, _P],
    "md2_hat_fwd": [c_void, _P, _P, _I32, _P],
    "md2_hat_bwd": [c_void, _P, _P, _I32, _P],
    "md2_compose_T_fwd": [c_void, _P, _P, _I32, _P, _P, _I32, _P],
    "md2_compose_T_bwd": [c_void, _P, _P, _I32, _P, _P, _P, _P, _I32, _P],
    "md2_grid_sample_fwd": [c_void, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_grid_sample_bwd": [c_void, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_upsample_bilinear_fwd": [c_void, _P, _P, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_upsample_bilinear_bwd": [c_void, _P, _P, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_ssim_fwd": [c_void, _P, _P, _P, _I32, _I32, _I32, _I32, _P],
    "md2_ssim_bwd": [c_void, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _P],
    "md2_photometric_min_fwd": [c_void, _I32, C.POINTER(_P), C.POINTER(_I64), _P, _I64, _P, _F, _P, _P,
                                _I32, _I32, _I32, _I32, _P],
    "md2_photometric_min_bwd": [c_void, _I32, C.POINTER(_P), C.POINTER(_I64), _P, _I64, _P, _F, _P, _P,
                                C.POINTER(_P), _P, _P, _I32, _I32, _I32, _I32, _P],
    "md2_smooth_loss_fwd": [c_void, _P, _P, _I64, _P, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_smooth_loss_bwd": [c_void, _P, _P, _I64, _F, _P, _P, _I32, _I32, _I32, _I32, _I32, _P],
    "md2_view_synthesis_loss_fwd": [c_void, C.POINTER(VslDesc), _P],
    "md2_view_synthesis_loss_bwd": [c_void, C.POINTER(VslDesc), _F, _P],
    "md2_view_synthesis_loss_fwdbwd": [c_void, C.POINTER(VslDesc), _F, _P],
    "md2_view_synthesis_loss_fwdbwd_host": [c_void, C.POINTER(VslDesc), _F, _I32],
    "md2_view_synthesis_loss_fwdbwd_host_submit": [c_void, C.POINTER(VslDesc), _F, _I32, _I32],
    "md2_host_wait": [c_void, _I32],
    "md2_warp_fwd": [c_void, C.POINTER(VslDesc), C.POINTER(_P), _P],
    "md2_warp_bwd": [c_void, C.POINTER(VslDesc), C.POINTER(_P), _P],
    "md2_adam_step": [c_void, _I32, C.POINTER(_P), C.POINTER(_P), C.POINTER(_I64), _P, _P, _F, _F, _F, _F, _F, _P],
    "md2_slow_depth": [c_void, C.POINTER(VslDesc), _I32, _F, _F, _F, _F, _P, _P, _P, _I64, _P],
}
ADAM_MAX_TENSORS = 16
EXPORTS = ["md2_version", "md2_last_error", "md2_launch_count"] + list(_SIGS)

_lib = None
_lock = threading.Lock()


class Md2Error(RuntimeError):
    pass


def load_library(path=LIB_PATH):
    """dlopen the C-ABI library and declare its signatures (no GPU needed for this)."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(path):
            raise Md2Error(f"{path} is missing: build it first (python -c 'import __graft_entry__ as g; g.build()'). "
                           "There is no CPU fallback.")
        lib = C.CDLL(path)
        lib.md2_version.restype = C.c_char_p
        lib.md2_last_error.restype = C.c_char_p
        lib.md2_launch_count.restype = C.c_int64
        lib.md2_launch_count.argtypes = [c_void]
        for name, args in _SIGS.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int
        _lib = lib
        return lib


class Context:
    """md2_ctx wrapper: one per (process, device)."""
    _by_device: dict = {}

    def __init__(self, device_index):
        if not torch.cuda.is_available():
            raise Md2Error("monodepth2.jl_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.lib = load_library()
        self.device = device_index
        h = c_void()
        self._check(self.lib.md2_create(device_index, C.byref(h)))
        self.handle = h

    @classmethod
    def get(cls, device):
        idx = device.index if device.index is not None else torch.cuda.current_device()
        ctx = cls._by_device.get(idx)
        if ctx is None:
            ctx = cls._by_device[idx] = Context(idx)
        return ctx

    def _check(self, status):
        if status != 0:
            raise Md2Error(self.lib.md2_last_error().decode())

    def call(self, name, *args):
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._check(getattr(self.lib, name)(self.handle, *args, stream))

    @property
    def launches(self):
        return int(self.lib.md2_launch_count(self.handle))

    def profile(self, on):
        self._check(self.lib.md2_profile_enable(self.handle, int(on)))

    def profile_read_phases(self):
        a, b, c, n = C.c_float(), C.c_float(), C.c_float(), C.c_int64()
        self._check(self.lib.md2_profile_read_phases(self.handle, C.byref(a), C.byref(b), C.byref(c), C.byref(n)))
        return a.value, b.value, c.value, n.value

    def profile_read(self):
        ms, n = C.c_float(), C.c_int64()
        self._check(self.lib.md2_profile_read(self.handle, C.byref(ms), C.byref(n)))
        return ms.value, n.value


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise Md2Error("monodepth2.jl_b200 operators take CUDA tensors only (no CPU fallback)")
