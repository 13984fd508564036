"""Test helper: the two float64 oracles with a camera per image and with gradients with respect to K and invK.

torch oracle: oracle/torch_oracle.py with K and invK as independent autograd leaves.  c oracle: oracle/c_oracle.c for the
value and the other gradients, tests/c_oracle_intrinsics.c for the hand-derived reverse pass to K and invK.  A camera per
image is evaluated image by image: the path is independent per image, and every mean of the loss is over the images, so
the batch loss is the mean of the per-image losses and the gradients of image n are 1/N of its own."""
import ctypes as C
import os
import subprocess
import tempfile

import torch

from oracle import c_oracle as CO
from oracle import torch_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "c_oracle_intrinsics.c")
_lib = None


def _build():
    """compiled into a per-user temporary directory (the tree may be read-only)"""
    out = os.path.join(tempfile.gettempdir(), f"md2_test_{os.getuid()}")
    os.makedirs(out, exist_ok=True)
    so = os.path.join(out, "libc_oracle_intrinsics.so")
    deps = [SRC, os.path.join(os.path.dirname(HERE), "oracle", "c_oracle.c")]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        tmp = so + f".{os.getpid()}"
        subprocess.run(["gcc", "-O2", "-std=c99", "-fPIC", "-fvisibility=hidden", "-ffp-contract=off", "-shared", "-o", tmp, SRC, "-lm"],
                       check=True)
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(_build())
        _lib.co_vsl_intrinsics_grad.restype = C.c_int
    return _lib


def _images(K, N):
    """(3,3) -> None (one camera); (N,3,3) -> the list of per-image matrices"""
    return None if K.dim() == 2 else [K[n] for n in range(N)]


def _slice(x, disps, rv, tv, auto, choices, n):
    return (x[n:n + 1], [d[n:n + 1] for d in disps], [r[n:n + 1] for r in rv], [t[n:n + 1] for t in tv],
            None if auto is None else auto[n:n + 1], None if choices is None else choices[:, n:n + 1])


def torch_loss(x, disps, rv, tv, K, invK, *, choices=None, auto=None, **kw):
    """float64 torch-oracle loss (forced when `choices` is given); K / invK (3,3) or (N,3,3), differentiable"""
    def one(x, disps, rv, tv, K, invK, auto, choices):
        if choices is None:
            return O.view_synthesis_loss(x, disps, rv, tv, K, invK, automasking=auto is not None, auto_loss=auto, **kw)
        return O.view_synthesis_loss_forced(x, disps, rv, tv, K, invK, choices, auto_loss=auto, **kw)
    N = x.shape[0]
    if K.dim() == 2:
        return one(x, disps, rv, tv, K, invK, auto, choices)
    return sum(one(*_slice(x, disps, rv, tv, auto, choices, n)[:4], K[n], invK[n], *_slice(x, disps, rv, tv, auto, choices, n)[4:])
               for n in range(N)) / N


def _kgrad(x, disps, rv, tv, K, invK, auto, choices, target_id, source_ids, min_depth, max_depth, alpha):
    f64 = lambda t: t.detach().to(torch.float64).contiguous()
    x = f64(x)
    N, L, Cc, H, W = x.shape
    ds = [f64(d) for d in disps]
    rv = torch.stack([f64(r) for r in rv]).contiguous()
    tv = torch.stack([f64(t) for t in tv]).contiguous()
    Kd, iKd = f64(K).reshape(3, 3).contiguous(), f64(invK).reshape(3, 3).contiguous()
    al = f64(auto).reshape(N, H, W).contiguous() if auto is not None else None
    ch = choices.detach().cpu().to(torch.int32).contiguous() if choices is not None else None
    gK, giK = torch.zeros(3, 3, dtype=torch.float64), torch.zeros(3, 3, dtype=torch.float64)
    D = C.POINTER(C.c_double)
    p = lambda t: C.cast(t.data_ptr(), D) if t is not None else None
    n = len(ds)
    ints = lambda v: (C.c_int * len(v))(*v)
    rc = lib().co_vsl_intrinsics_grad(
        p(x), N, L, Cc, H, W, n, (D * n)(*[p(d) for d in ds]), ints([d.shape[-2] for d in ds]), ints([d.shape[-1] for d in ds]),
        p(rv), p(tv), p(Kd), p(iKd), int(target_id), len(source_ids), ints(list(source_ids)), C.c_double(min_depth),
        C.c_double(max_depth), p(al), C.c_double(alpha), C.cast(ch.data_ptr(), C.POINTER(C.c_int)) if ch is not None else None,
        p(gK), p(giK))
    assert rc == 0
    return gK, giK


def c_vsl(x, disps, rv, tv, K, invK, *, auto=None, choices=None, export_choices=False, target_id=1, source_ids=(0, 2),
          min_depth=0.1, max_depth=100.0, alpha=0.85):
    """C-oracle value and gradients (dict as oracle.c_oracle.view_synthesis_loss, plus gK / ginvK of the shape of K)"""
    kw = dict(target_id=target_id, source_ids=source_ids, min_depth=min_depth, max_depth=max_depth)
    N = x.shape[0]
    if K.dim() == 2:
        out = CO.view_synthesis_loss(x, disps, rv, tv, K, invK, auto_loss=auto, choices=choices, export_choices=export_choices,
                                     alpha=alpha, **kw)
        out["gK"], out["ginvK"] = _kgrad(x, disps, rv, tv, K, invK, auto, choices, alpha=alpha, **kw)
        return out
    parts = [c_vsl(*_slice(x, disps, rv, tv, auto, choices, n)[:4], K[n], invK[n], auto=_slice(x, disps, rv, tv, auto, choices, n)[4],
                   choices=_slice(x, disps, rv, tv, auto, choices, n)[5], export_choices=export_choices, alpha=alpha, **kw)
             for n in range(N)]
    out = {"loss": sum(q["loss"] for q in parts) / N,
           "gdisp": [torch.cat([q["gdisp"][l] for q in parts]) / N for l in range(len(disps))],
           "grvec": [torch.cat([q["grvec"][s] for q in parts]) / N for s in range(len(source_ids))],
           "gtvec": [torch.cat([q["gtvec"][s] for q in parts]) / N for s in range(len(source_ids))],
           "gK": torch.stack([q["gK"] for q in parts]) / N, "ginvK": torch.stack([q["ginvK"] for q in parts]) / N}
    if export_choices:
        out["choices"] = torch.cat([q["choices"] for q in parts], 1)
    return out
