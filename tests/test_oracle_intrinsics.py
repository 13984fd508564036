"""Gradients with respect to the camera intrinsics K and invK (shared or per image) in the two float64 oracles: the
hand-derived reverse pass of tests/c_oracle_intrinsics.c against torch autograd, both against central finite differences,
and the per-image form against the shared one.  K and invK are independent inputs throughout, as in the reference."""
import pytest
import torch

from intrinsics_oracle import c_vsl, torch_loss
from oracle import torch_oracle as O

F64 = torch.float64


def cameras(N, W, H, seed):
    """distinct per-image K (focal 0.5-0.9 W, principal point within +-10 px of the centre) and their inverses"""
    g = torch.Generator().manual_seed(seed)
    f = (0.5 + 0.4 * torch.rand(N, 2, generator=g, dtype=F64)) * W
    c = torch.tensor([W / 2.0, H / 2.0], dtype=F64) + (torch.rand(N, 2, generator=g, dtype=F64) - 0.5) * 20
    K = torch.zeros(N, 3, 3, dtype=F64)
    K[:, 0, 0], K[:, 1, 1], K[:, 0, 2], K[:, 1, 2], K[:, 2, 2] = f[:, 0], f[:, 1], c[:, 0], c[:, 1], 1.0
    return K, torch.linalg.inv(K)


def batch(N, C, H, W, seed, sigma=0.01):
    x, disps, rv, tv = O.synthetic_batch(N, C, H, W, seed=seed, pose_sigma=sigma, dtype=F64)
    return x, disps, rv, tv


def torch_grads(x, disps, rv, tv, K, invK, auto=None, choices=None):
    Kd, iKd = K.clone().requires_grad_(True), invK.clone().requires_grad_(True)
    loss = torch_loss(x, disps, rv, tv, Kd, iKd, auto=auto, choices=choices)
    gK, giK = torch.autograd.grad(loss, (Kd, iKd))
    return loss.item(), gK, giK


def per_matrix_err(a, b):
    a, b = a.reshape(-1, 3, 3), b.reshape(-1, 3, 3)
    return max(((a[m] - b[m]).abs().max() / b[m].abs().max()).item() for m in range(a.shape[0]))


CASES = [  # N, C, H, W, automask, per_image, pose sigma
    pytest.param(2, 1, 20, 28, False, False, 0.01, id="shared"),
    pytest.param(2, 3, 18, 26, True, True, 0.01, id="per-image-automask"),
    pytest.param(3, 1, 17, 23, False, True, 0.3, id="per-image-points-leave-the-image"),
]


@pytest.mark.parametrize("N,C,H,W,am,per_image,sigma", CASES)
def test_c_oracle_matches_torch_autograd(N, C, H, W, am, per_image, sigma):
    x, disps, rv, tv = batch(N, C, H, W, seed=N + H, sigma=sigma)
    K, invK = cameras(N, W, H, seed=W) if per_image else O.make_K(W, H, dtype=F64)
    auto = O.automasking_loss(O.SSIM(), x, x[:, 1], (0, 2)) if am else None
    co = c_vsl(x, disps, rv, tv, K, invK, auto=auto, export_choices=True)
    # the torch oracle with the C oracle's own decisions: the same piece of the piecewise-smooth loss, exactly
    loss, gK, giK = torch_grads(x, disps, rv, tv, K, invK, auto=auto, choices=co["choices"])
    assert abs(co["loss"] - loss) <= 1e-12 * abs(loss)
    assert co["gK"].shape == K.shape and co["ginvK"].shape == invK.shape
    assert per_matrix_err(co["gK"], gK) <= 1e-12
    assert per_matrix_err(co["ginvK"], giK) <= 1e-12


def test_both_sources_inverted_and_points_behind_the_camera():
    """large poses send points out of the image and some behind the camera plane; both sources precede the target, so
    composeT inverts both poses"""
    N, C, H, W = 2, 1, 16, 24
    x, disps, rv, tv = batch(N, C, H, W, seed=4, sigma=0.6)
    K, invK = cameras(N, W, H, seed=3)
    kw = dict(target_id=2, source_ids=(0, 1))
    co = c_vsl(x, disps, rv, tv, K, invK, export_choices=True, **kw)
    Kd, iKd = K.clone().requires_grad_(True), invK.clone().requires_grad_(True)
    loss = torch_loss(x, disps, rv, tv, Kd, iKd, choices=co["choices"], **kw)
    gK, giK = torch.autograd.grad(loss, (Kd, iKd))
    assert per_matrix_err(co["gK"], gK) <= 1e-12
    assert per_matrix_err(co["ginvK"], giK) <= 1e-12


@pytest.mark.parametrize("per_image,forced", [(False, False), (False, True), (True, True)])
def test_finite_differences(per_image, forced):
    N, C, H, W = 2, 1, 14, 20
    x, disps, rv, tv = batch(N, C, H, W, seed=9)
    K, invK = cameras(N, W, H, seed=5) if per_image else O.make_K(W, H, dtype=F64)
    co = c_vsl(x, disps, rv, tv, K, invK, export_choices=True)
    ch = co["choices"] if forced else None
    f = lambda K_, iK_: c_vsl(x, disps, rv, tv, K_, iK_, choices=ch)["loss"]
    g = torch.Generator().manual_seed(2)
    for which in range(2):
        for _ in range(2):
            d = torch.randn(K.shape, generator=g, dtype=F64)
            d[..., 2, :] = 0.0                      # keep the last row (0, 0, 1) of K, the first two of invK are free too
            # (steps that move the projected points by ~1e-4 px: the loss is strongly curved in invK)
            eps = 1e-6 * K.abs().max().item() if which == 0 else 1e-8
            if which == 0:
                fd = (f(K + eps * d, invK) - f(K - eps * d, invK)) / (2 * eps)
                an = (co["gK"] * d).sum().item()
            else:
                fd = (f(K, invK + eps * d) - f(K, invK - eps * d)) / (2 * eps)
                an = (co["ginvK"] * d).sum().item()
            assert abs(fd - an) <= 1e-5 * max(abs(an), 1e-12) + 1e-10, (which, fd, an)


def test_identical_per_image_copies_equal_shared():
    N, C, H, W = 3, 3, 16, 22
    x, disps, rv, tv = batch(N, C, H, W, seed=6)
    K, invK = O.make_K(W, H, dtype=F64)
    a = c_vsl(x, disps, rv, tv, K, invK)
    b = c_vsl(x, disps, rv, tv, K.expand(N, 3, 3), invK.expand(N, 3, 3))
    assert abs(a["loss"] - b["loss"]) <= 1e-13 * abs(a["loss"])
    for name in ("gK", "ginvK"):
        assert per_matrix_err(b[name].sum(0), a[name]) <= 1e-13
    for u, v in zip(a["gdisp"] + a["grvec"] + a["gtvec"], b["gdisp"] + b["grvec"] + b["gtvec"]):
        assert ((u - v).abs().max() / v.abs().max()).item() <= 1e-13
