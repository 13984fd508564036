"""Row F1 on the GPU: the training step around the loss (src/Monodepth.jl:156-176) -- stand-in model -> fused loss ->
backward -> [bucketed NCCL all-reduce] -> fused ADAM; visualisation copies on a side stream; checkpoint / resume."""
import os
import socket

import pytest
import torch

import monodepth2_jl_b200 as M
from oracle import torch_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _strict_fp32_deterministic_convs():
    """the stand-in networks are the host framework's: pin cuDNN to fp32 (no TF32) and deterministic algorithms so that two
    runs of the same model see the same gradients (ADAM's sign-like early steps amplify any difference to +-lr)"""
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = False, True, False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = old


def dev():
    return torch.device("cuda", 0)


def batch(n, c, h, w, seed):
    x, _, _, _ = O.synthetic_batch(n, c, h, w, seed=seed)
    return x.to(dev())


def test_step_trains_and_matches_autograd_plus_torch_adam():
    """the trainer's gradient (flat buffer, hooks) == torch.autograd's on an identical model, its first update == the
    Flux rule applied to that gradient, and three steps stay within ADAM's step bound of torch.optim.Adam (the two rules
    coincide; early steps are sign-like, so elements whose gradient is rounding noise may step the other way)"""
    W, H = 128, 64
    trainer, model, cache, hp = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, seed=3)
    torch.manual_seed(3)
    ref_model = M.StandInModel(3).to(dev()).train()
    ref_model.load_state_dict(model.state_dict())
    ref_opt = torch.optim.Adam(ref_model.parameters(), lr=1e-4, eps=1e-8)
    x = batch(2, 3, H, W, 1)
    p0 = trainer.flat.data.clone()
    losses = []
    for it in range(3):
        loss, _ = trainer.step(x)
        losses.append(loss.item())
        ref_opt.zero_grad()
        l2, *_ = M.train_loss(ref_model, x, None, cache, hp, False)
        l2.backward()
        if it == 0:
            assert abs(l2.item() - loss.item()) <= 1e-6 * abs(l2.item())
            for (n1, p1), (_, p2) in zip(model.named_parameters(), ref_model.named_parameters()):
                if p2.grad is None:
                    continue
                scale = p2.grad.abs().max().clamp_min(1e-12)
                assert ((p1.grad - p2.grad).abs().max() / scale).item() <= 2e-3, n1          # (cuDNN picks its algorithms per call)
            g = trainer.flat.grad.double().cpu()
            upd = 1e-4 * (0.1 * g / (1 - 0.9)) / ((0.001 * g * g / (1 - 0.999)).sqrt() + 1e-8)     # Flux ADAM, t = 1
            assert torch.allclose((p0.double().cpu() - upd).float(), trainer.flat.data.cpu(), rtol=1e-5, atol=1e-8)
        ref_opt.step()
    assert all(torch.isfinite(torch.tensor(losses)))
    assert trainer.opt.steps == 3
    close, total = 0, 0
    for (n1, p1), (n2, p2) in zip(model.named_parameters(), ref_model.named_parameters()):
        assert n1 == n2
        assert (p1 - p2).abs().max().item() <= 2 * 1e-4 * 3 + 1e-6, n1
        close += torch.isclose(p1, p2, rtol=1e-4, atol=3e-6).sum().item(); total += p1.numel()
    assert close / total > 0.9, close / total
    assert losses[-1] != losses[0]


def test_visualisation_ticket_and_automasking():
    W, H = 128, 64
    trainer, model, cache, hp = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, automasking=True, seed=1)
    x = batch(2, 3, H, W, 2)
    loss, ticket = trainer.step(x, do_visualization=True)
    vd, vw, vl = ticket.get()
    assert not vd.is_cuda and vd.shape == (2, 1, H, W) and len(vw) == 2 and vw[0].shape == (2, 3, H, W) and vl.shape == (2, 1, H, W)
    assert vd.is_pinned() and torch.isfinite(vl).all() and 0.0 <= vd.min() and vd.max() <= 1.0
    # the warp-loss map of the step averages to its photometric share of the loss: mean(vis_loss) is what src/training.jl:66 adds
    assert 0.0 < vl.mean().item() < loss.item() * 4 * 1.5


def test_checkpoint_resume_continues_the_same_trajectory(tmp_path):
    W, H = 128, 64
    xs = [batch(2, 3, H, W, 10 + k) for k in range(5)]
    a, ma, _, _ = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, seed=5)
    for k in range(3):
        a.step(xs[k])
    path = str(tmp_path / "ckpt.pt")
    a.save_checkpoint(path)                    # model + ADAM moments + step counter
    for k in range(3, 5):
        a.step(xs[k])
    b, mb, _, _ = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, seed=99)    # different initial weights
    b.load_checkpoint(path)
    assert b.steps == 3 and b.opt.steps == 3
    for k in range(3, 5):
        b.step(xs[k])
    frac = lambda m1, m2: sum(torch.isclose(p1, p2, rtol=1e-4, atol=2e-6).sum().item() for p1, p2 in zip(m1.parameters(), m2.parameters())) / \
        sum(p.numel() for p in m1.parameters())
    assert frac(ma, mb) > 0.9
    # a cold optimiser (what resuming from the reference's model-only BSON dump does) does NOT reproduce the trajectory
    c, mc, _, _ = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, seed=99)
    sd = torch.load(path, map_location="cpu", weights_only=False)
    with torch.no_grad():
        mc.load_state_dict(sd["model"])
    for k in range(3, 5):
        c.step(xs[k])
    assert frac(ma, mc) < 0.6


def _nccl_worker(rank, world, port, q):
    try:
        _nccl_worker_body(rank, world, port, q)
    except Exception as e:      # the parent must not sit in q.get until its timeout
        import traceback
        q.put((rank, "error: " + repr(e) + "\n" + traceback.format_exc(), None))
        raise


def _nccl_worker_body(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    d = torch.device("cuda", rank)
    torch.cuda.set_device(d)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=d)
    from monodepth2_jl_b200 import dist as D
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = False, True, False
    W, H, NB = 128, 64, 4
    x, _, _, _ = O.synthetic_batch(NB, 3, H, W, seed=31)
    xs = D.shard_batch(x, rank, world).to(d)
    res = {}
    for overlap in (True, False):
        trainer, model, _, _ = M.make_training_setup(W, H, d, channels=3, batch_size=NB, seed=7, overlap=overlap, bucket_bytes=1 << 20)
        for m in model.modules():               # batch statistics are per rank (as in any data-parallel BatchNorm): freeze them
            if isinstance(m, torch.nn.BatchNorm2d):
                m.eval()
        loss, _ = trainer.step(xs)
        res[overlap] = (trainer.flat.grad.cpu().numpy().copy(), trainer.flat.data.cpu().numpy().copy(), float(D.global_loss(loss, xs.shape[0])),
                        len(trainer.flat.buckets), trainer.flat.calls)
    g = [torch.full((3,), float(rank + 1), device=d)]
    D.allreduce_mean_(g)
    q.put((rank, res, g[0].cpu().tolist()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_step_equals_the_full_batch_step():
    """data-parallel step over NCCL at world size 2: the all-reduced gradient (sum over ranks x 1/2) and the updated
    parameters equal those of ONE process stepping on the whole batch; overlapped and blocking all-reduce agree"""
    import numpy as np
    import torch.multiprocessing as mp
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = []
    for _ in range(2):
        r = q.get(timeout=240)
        assert not isinstance(r[1], str), r[1]
        res.append(r)
    res.sort(key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    W, H, NB = 128, 64, 4
    x, _, _, _ = O.synthetic_batch(NB, 3, H, W, seed=31)
    full, model, _, _ = M.make_training_setup(W, H, dev(), channels=3, batch_size=NB, seed=7)
    for m in model.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eval()
    loss, _ = full.step(x.to(dev()))
    gfull, pfull = full.flat.grad.cpu().numpy(), full.flat.data.cpu().numpy()
    for rank, r, shared in res:
        assert shared == [1.5, 1.5, 1.5]
        for overlap in (True, False):
            g, p, gl, nb, calls = r[overlap]
            assert nb >= 4 and calls == nb
            assert abs(gl - loss.item()) <= 1e-5 * abs(loss.item())
            assert np.abs(0.5 * g - gfull).max() <= 2e-4 * np.abs(gfull).max()
            assert np.abs(p - pfull).max() <= 2.5e-4          # (ADAM's first step is +-lr per element: sign flips of ~0 gradients)
            assert (np.abs(p - pfull) < 1e-6).mean() > 0.98
        assert np.allclose(r[True][0], r[False][0], rtol=1e-4, atol=1e-7 * np.abs(gfull).max())    # overlapped == blocking all-reduce


def test_training_reduces_the_loss_on_a_fixed_batch():
    """the whole stack end to end: 40 steps of the trainer on one batch must lower the loss (gradient signs / scaling through
    the stand-in networks, the fused loss, the flat gradient buffer and the fused ADAM)"""
    W, H = 128, 64
    trainer, model, cache, hp = M.make_training_setup(W, H, dev(), channels=3, batch_size=2, seed=11, lr=1e-3)
    x = batch(2, 3, H, W, 5)
    losses = [trainer.step(x)[0].item() for _ in range(40)]
    assert all(l == l for l in losses)
    assert min(losses[-5:]) < 0.99 * losses[0] and sum(losses[-5:]) / 5 < losses[0], (losses[0], losses[-5:])


def test_profile_phases_of_a_step():
    x, disps, rv, tv = O.synthetic_batch(2, 1, 64, 128, seed=3)
    from oracle.torch_oracle import make_K
    K, invK = make_K(128, 64)
    d = dev()
    ctx = M.Context.get(d)
    args = (x.to(d), [t.to(d).requires_grad_(True) for t in disps], [t.to(d) for t in rv], [t.to(d) for t in tv], K.to(d), invK.to(d))
    ctx.profile(2)
    try:
        for _ in range(3):
            M.view_synthesis_loss(*args)
        prep, march, finish, n = ctx.profile_read_phases()
    finally:
        ctx.profile(False)
    assert n == 3 and prep > 0 and march > 0 and finish > 0
