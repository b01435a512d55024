"""2-GPU (NCCL) check of the data-parallel path: the generator gradients produced by two ranks, each holding one sample and
relying on the AUTOMATIC reduction of sync_batchnorm.DataParallelWithCallback (hooks; no explicit reduce call — the pattern of
train_generator.py:314-322), equal the gradients of a single process on the concatenated batch of two, and so does the loss.
Skipped on machines with fewer than 2 GPUs."""
import os
import socket
import sys

import pytest
import torch
import torch.multiprocessing as mp

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import hrv_loader  # noqa: E402

hrv_loader.load()

pytestmark = pytest.mark.gpu
H = W = 256
SEED = 29


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _build(dev):
    import network_generator
    from helpers import gen_opt, synth_state_dict
    m = network_generator.SPADEGenerator(gen_opt(H, W, True), 9)
    m.load_state_dict(synth_state_dict("gen", SEED))
    return m.to(dev).train()


def _loss_and_grads(m, x, seg, R, noise_slice):
    from hrviton_b200 import synth
    cnt = [0]

    def noise(b, hh, ww):
        t = synth.spade_noise(2, hh, ww, SEED, cnt[0])[noise_slice].to(x.device)
        cnt[0] += 1
        return t

    (m.module if hasattr(m, "module") else m).noise_source = noise
    out = m(x, seg)
    loss = (out * R).mean()
    loss.backward()
    torch.cuda.synchronize()
    return float(loss)


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE=str(world), RANK=str(rank), LOCAL_RANK=str(rank))
    torch.cuda.set_device(rank)
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    from hrviton_b200 import ddp, synth
    m = _build("cuda")
    if rank == 1:  # replicas deliberately start different: wrapping must broadcast rank 0's parameters and buffers
        with torch.no_grad():
            for p in m.parameters():
                p.add_(0.01)
    w = ddp.DataParallelWithCallback(m, device_ids=[rank])
    x, seg = synth.gen_inputs(2, H, W, SEED)
    R = synth.normalish((2, 3, H, W), SEED, "lossw")
    sl = slice(rank, rank + 1)
    loss = _loss_and_grads(w, x[sl].cuda(), seg[sl].cuda(), R[sl].cuda(), sl)
    ret[rank] = (loss, {n: p.grad.detach().cpu() for n, p in m.named_parameters() if p.grad is not None}, w._reducer.launched,
                 {n: b.detach().cpu() for n, b in m.named_buffers()})
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_ranks_equal_one_process_on_the_concatenated_batch():
    from hrviton_b200 import synth
    world = 2
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    (l0, g0, n0, b0), (l1, g1, n1, b1) = ret[0], ret[1]
    assert n0 == n1 and n0 >= 1
    for k in g0:
        assert torch.equal(g0[k], g1[k]), k  # both ranks hold the same averaged gradient
    # single process, batch of two
    torch.cuda.set_device(0)
    m = _build("cuda")
    x, seg = synth.gen_inputs(2, H, W, SEED)
    R = synth.normalish((2, 3, H, W), SEED, "lossw")
    loss = _loss_and_grads(m, x.cuda(), seg.cuda(), R.cuda(), slice(0, 2))
    assert abs(0.5 * (l0 + l1) - loss) < 1e-5 * max(1.0, abs(loss)), (l0, l1, loss)
    for k, b in m.named_buffers():  # spectral-norm u/v after the power iteration: identical (same weights everywhere)
        assert torch.allclose(b.detach().cpu(), b0[k], atol=1e-6) and torch.equal(b0[k], b1[k]), k
    worst = 0.0
    for name, p in m.named_parameters():
        if p.grad is None:
            assert name not in g0
            continue
        ref = p.grad.detach().cpu()
        # mean over 2 samples = average of the per-rank means; per-sample arithmetic is identical (InstanceNorm, per-sample noise),
        # only the fp32 accumulation order of the weight-gradient split-K differs
        rel = float((g0[name] - ref).norm() / (ref.norm() + 1e-20))
        worst = max(worst, rel)
        assert rel < 2e-3 or float(ref.norm()) < 1e-6, (name, rel)
    print("MULTIGPU 2 ranks vs 1 process: loss %.6f vs %.6f, worst per-parameter gradient rel diff %.3e, %d bucket all-reduces" % (0.5 * (l0 + l1), loss, worst, n0))
