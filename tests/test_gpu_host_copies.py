"""Host-buffer entry point (md2_view_synthesis_loss_fwdbwd_host / _submit / md2_host_wait): what it copies back.

The call moves the outputs of the device mirror to the caller's host arrays.  With one image group, disparity-gradient
arrays that lie back to back in host memory travel as ONE device-to-host copy of the whole stretch.  The call must never
write a host byte outside the output arrays of the descriptor: arrays separated by a gap (separate allocations that happen
to lie close together, or a caller's own padding) take one copy per array, and the gaps keep their contents."""
import ctypes as C

import pytest
import torch

import monodepth2_jl_b200 as M
from monodepth2_jl_b200 import _lib as L
from oracle import torch_oracle as O

pytestmark = pytest.mark.gpu

SENTINEL = 0x7FC0BEEF           # a NaN payload that neither the kernels nor uninitialised device memory produce
GAPS = (8, 100, 1000)           # floats between disparity-gradient arrays l and l+1 (at most 1024: the old one-copy bound)
MARGIN = 64                     # sentinel floats before the first and after the last array


def dev():
    return torch.device("cuda", 0)


def pinned(*shape):
    return torch.zeros(*shape, dtype=torch.float32).pin_memory()


def device_path(x, disps, rv, tv, K, invK, scales):
    d = dev()
    dg = [t.to(d).requires_grad_(True) for t in disps]
    rg = [t.to(d).requires_grad_(True) for t in rv]
    tg = [t.to(d).requires_grad_(True) for t in tv]
    loss = M.view_synthesis_loss(x.to(d), dg, rg, tg, K.to(d), invK.to(d), scales=scales)
    loss.backward()
    return loss.item(), [t.grad.cpu() for t in dg], [t.grad.cpu() for t in rg], [t.grad.cpu() for t in tg]


class GappedCall:
    """every input in pinned host memory, the L disparity-gradient arrays carved out of ONE pinned buffer with GAPS
    between them, every float outside the arrays set to SENTINEL"""

    def __init__(self, x, disps, rv, tv, K, invK, scales):
        N, _, Cc, H, W = x.shape
        # (the inputs share one pinned allocation, as in HostViewSynthesisLoss: the input direction stays on its usual route)
        ins = [x] + list(disps)
        offs, tot = [], 0
        for t in ins:
            offs.append(tot); tot += (t.numel() + 63) // 64 * 64
        self.in_buf = pinned(tot)
        views = [self.in_buf[o:o + t.numel()].view(t.shape) for o, t in zip(offs, ins)]
        for a, b in zip(views, ins):
            a.copy_(b)
        self.x, self.disps = views[0], views[1:]
        self.rv = [pinned(N, 3) for _ in rv]
        self.tv = [pinned(N, 3) for _ in tv]
        for a, b in zip(self.rv + self.tv, rv + tv):
            a.copy_(b)
        self.K, self.invK = K.t().contiguous().pin_memory(), invK.t().contiguous().pin_memory()
        sizes = [t.numel() for t in disps]
        gaps = [GAPS[l % len(GAPS)] for l in range(len(disps) - 1)]
        self.buf = pinned(MARGIN + sum(sizes) + sum(gaps) + MARGIN)
        self.buf.view(torch.int32).fill_(SENTINEL)
        self.gd, self.owned, o = [], torch.zeros(self.buf.numel(), dtype=torch.bool), MARGIN
        for l, (n, t) in enumerate(zip(sizes, disps)):
            self.gd.append(self.buf[o:o + n].view(t.shape))
            self.owned[o:o + n] = True
            o += n + (gaps[l] if l < len(gaps) else 0)
        self.gr = [pinned(N, 3) for _ in rv]
        self.gt = [pinned(N, 3) for _ in tv]
        self.loss = pinned(1)
        self.desc = L.make_vsl_desc(
            target=self.x[:, 1], target_stride=self.x.stride(0), sources=[self.x[:, 0], self.x[:, 2]],
            source_strides=[self.x.stride(0)] * 2, disparities=self.disps, K_cm=self.K, invK_cm=self.invK,
            rot=self.rv, trans=self.tv, pose_mode=1, invert=[1, 0], smooth_weight=[1e-3 * s for s in scales],
            loss_scale=1.0 / len(disps), loss=self.loss, grad_disparity=self.gd, grad_rot=self.gr, grad_trans=self.gt,
            shape=(N, Cc, H, W))

    def gap_words(self):
        return self.buf.view(torch.int32)[~self.owned]

    def check(self, ref, tag):
        words = self.gap_words()
        bad = (words != SENTINEL).nonzero().flatten()
        assert bad.numel() == 0, (tag, f"{bad.numel()} of {words.numel()} floats outside the gradient arrays overwritten")
        rl, rgd, rgr, rgt = ref
        assert abs(self.loss.item() - rl) <= 2e-6 * max(1.0, abs(rl)), (tag, self.loss.item(), rl)
        for l, (a, b) in enumerate(zip(self.gd, rgd)):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-9), (tag, "gdisp", l)
        for a, b in zip(self.gr + self.gt, rgr + rgt):
            assert torch.allclose(a, b, rtol=1e-4, atol=1e-8), (tag, "pose")


def _batch(seed=21):
    N, Cc, H, W = 2, 3, 48, 96
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, seed=seed)
    K, invK = O.make_K(W, H)
    return x, disps, rv, tv, K, invK, (0.125, 0.25, 0.5, 1.0)


def test_gaps_between_gradient_arrays_are_not_written():
    """one image group: separately placed gradient arrays 8, 100 and 1000 floats apart.  The gaps keep the sentinel and
    the gradients equal the device-pointer call; twice, so that the replayed graph is checked too."""
    x, disps, rv, tv, K, invK, scales = _batch()
    ref = device_path(x, disps, rv, tv, K, invK, scales)
    g = GappedCall(x, disps, rv, tv, K, invK, scales)
    ctx = M.Context.get(dev())
    for rep in range(2):
        if ctx.lib.md2_view_synthesis_loss_fwdbwd_host(ctx.handle, C.byref(g.desc), 1.0, 1):
            raise M.Md2Error(ctx.lib.md2_last_error().decode())
        g.check(ref, f"call {rep}")


def test_gaps_between_gradient_arrays_are_not_written_on_lanes():
    """the same through submit / wait on two lanes in flight at once (lanes own separate staging buffers and graphs)"""
    ctx = M.Context.get(dev())
    calls, refs = [], []
    for seed in (31, 32):
        x, disps, rv, tv, K, invK, scales = _batch(seed)
        refs.append(device_path(x, disps, rv, tv, K, invK, scales))
        calls.append(GappedCall(x, disps, rv, tv, K, invK, scales))
    for rep in range(2):
        for lane, g in zip((1, 2), calls):
            if ctx.lib.md2_view_synthesis_loss_fwdbwd_host_submit(ctx.handle, C.byref(g.desc), 1.0, 1, lane):
                raise M.Md2Error(ctx.lib.md2_last_error().decode())
        for lane, g, ref in zip((1, 2), calls, refs):
            if ctx.lib.md2_host_wait(ctx.handle, lane):
                raise M.Md2Error(ctx.lib.md2_last_error().decode())
            g.check(ref, f"lane {lane} call {rep}")


def test_wrapper_gradient_arrays_tile_exactly():
    """HostViewSynthesisLoss carves its disparity gradients back to back, so one image group keeps the one-copy route"""
    x, disps, rv, tv, K, invK, scales = _batch()
    N, _, Cc, H, W = x.shape
    hv = M.HostViewSynthesisLoss(N, Cc, H, W, [(d.shape[-1], d.shape[-2]) for d in disps], K, invK, device=dev(), groups=1,
                                 lanes=2)
    for grads in hv.lane_grads:
        g = grads["disparities"]
        for a, b in zip(g[:-1], g[1:]):
            assert b.data_ptr() == a.data_ptr() + 4 * a.numel()
        assert grads["_slab"].numel() == sum(t.numel() for t in g)


LAYOUTS = [
    pytest.param((1 / 16, 1 / 8, 1 / 4, 1 / 2, 1.0), id="five-scales"),
    pytest.param((1.0, 0.5, 0.25, 0.125), id="reversed"),
]


@pytest.mark.parametrize("groups", [1, 2])
@pytest.mark.parametrize("scales", LAYOUTS)
def test_wrapper_decoder_layouts_match_the_device_path(scales, groups):
    N, Cc, H, W = 3, 3, 64, 128
    x, disps, rv, tv = O.synthetic_batch(N, Cc, H, W, scales=scales, seed=23)
    K, invK = O.make_K(W, H)
    ref = device_path(x, disps, rv, tv, K, invK, scales)
    hv = M.HostViewSynthesisLoss(N, Cc, H, W, [(d.shape[-1], d.shape[-2]) for d in disps], K, invK, device=dev(),
                                 scales=scales, groups=groups)
    for rep in range(2):
        loss = hv(x, disps, rv, tv)
        rl, rgd, rgr, rgt = ref
        assert abs(loss - rl) <= 2e-6 * max(1.0, abs(rl)), (rep, loss, rl)
        for l, (a, b) in enumerate(zip(hv.grads["disparities"], rgd)):
            assert torch.allclose(a, b, rtol=1e-5, atol=1e-9), (rep, l)
        for a, b in zip(hv.grads["rvecs"] + hv.grads["tvecs"], rgr + rgt):
            assert torch.allclose(a, b, rtol=1e-4, atol=1e-8), rep
