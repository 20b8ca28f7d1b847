"""CPU, world_size 2, gloo: the host-side multi-process logic (column sharding, the single
loss+gradient all-reduce of the shared-parameter calibration step).  The kernels themselves need a GPU;
here the per-shard model is a small differentiable stand-in so that the collective path is what is tested."""
import os

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import lgar_b200
from lgar_b200 import parallel


def test_shard_range_covers_everything():
    for B in (1, 7, 32, 1000, 125_000):
        for world in (1, 2, 3, 8):
            spans = [parallel.shard_range(B, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == B
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, B, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.manual_seed(0)
    data = torch.arange(B, dtype=torch.float64) / B           # one "site" value per column
    lo, hi = parallel.shard_range(B, rank, world)
    p = [torch.nn.Parameter(torch.tensor([0.3, 0.7], dtype=torch.float64)), torch.nn.Parameter(torch.tensor(1.5, dtype=torch.float64))]
    opt = torch.optim.SGD(p, lr=0.1)
    ens = lambda ps: (ps[0][0] * data[lo:hi] + ps[0][1]) ** 2 * ps[1]
    loss_fn = lambda y: (y.sum(), hi - lo)
    loss = parallel.calibration_step(p, ens, loss_fn, opt)
    out[rank] = (float(loss), p[0].detach().numpy().copy(), float(p[1]))
    dist.destroy_process_group()


def test_calibration_step_world2_equals_single_process():
    B, port = 37, 29000 + os.getpid() % 2000
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, port, B, out), nprocs=2, join=True)
    # single-process reference
    data = torch.arange(B, dtype=torch.float64) / B
    p0 = torch.tensor([0.3, 0.7], dtype=torch.float64, requires_grad=True)
    p1 = torch.tensor(1.5, dtype=torch.float64, requires_grad=True)
    loss = (((p0[0] * data + p0[1]) ** 2) * p1).mean()
    loss.backward()
    want0 = (p0 - 0.1 * p0.grad).detach().numpy()
    want1 = float(p1 - 0.1 * p1.grad)
    for r in range(2):
        l, q0, q1 = out[r]
        assert abs(l - float(loss)) < 1e-12
        np.testing.assert_allclose(q0, want0, rtol=1e-12)
        assert abs(q1 - want1) < 1e-12


def _nan_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    data = torch.arange(8, dtype=torch.float64) / 8
    p = [torch.nn.Parameter(torch.tensor([0.3, 0.7], dtype=torch.float64)), torch.nn.Parameter(torch.tensor(1.5, dtype=torch.float64))]
    before = [q.detach().clone() for q in p]
    opt = torch.optim.SGD(p, lr=0.1)
    poison = float("nan") if rank == 1 else 1.0     # rank 1's shard produces a NaN gradient
    ens = lambda ps: (ps[0][0] * data + ps[0][1]) ** 2 * ps[1] * poison
    try:
        parallel.calibration_step(p, ens, lambda y: (y.sum(), 8), opt)
        out[rank] = "stepped"
    except RuntimeError as e:
        unchanged = all(torch.equal(q.detach(), b) for q, b in zip(p, before))
        out[rank] = ("raised", unchanged, all(q.grad is None for q in p), str(e))
    dist.destroy_process_group()


def test_calibration_step_refuses_a_nan_gradient_on_every_rank():
    port = 33000 + os.getpid() % 2000
    out = mp.Manager().dict()
    mp.spawn(_nan_worker, args=(2, port, out), nprocs=2, join=True)
    for r in range(2):
        assert out[r][:3] == ("raised", True, True), out[r]
