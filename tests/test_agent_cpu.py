"""CPU tests of the calibration agent's host logic (lgar_b200.agent, SURVEY 8f N2): the derived time configuration,
the loss functions and NSE against numbers worked out by hand from the reference's definitions, the mass-balance
report, checkpoint save / load, and the world-size-2 gloo gradient all-reduce.  The model is a small differentiable
stand-in with the dpLGAR surface (the kernels need a GPU: tests/test_gpu_agent.py)."""
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import lgar_b200
from lgar_b200 import agent as A

LB, UB = [0.0015, 1.0, 1e-6, 0.0], [0.015, 5.0, 30, 10.0]


def _cfg(endtime=48.0, subcycle=300.0, epochs=2, warmup=4):
    return dict(device="cpu", conversions=dict(hr_to_sec=3600.0, mm_to_cm=0.1),
                models=dict(endtime=endtime, subcycle_length=subcycle, forcing_resolution=3600.0,
                            hyperparameters=dict(warmup=warmup, epochs=epochs, learning_rate=1e-2, lb=LB, ub=UB)),
                data=dict())


class ToyModel(torch.nn.Module):
    """dpLGAR surface (alpha/n/ksat ParameterLists, ponded_depth_max, forward_record, set_internal_states)."""

    def __init__(self, L=3):
        super().__init__()
        P = lambda v: torch.nn.ParameterList([torch.nn.Parameter(torch.tensor(v + 0.1 * i, dtype=torch.float64)) for i in range(L)])
        self.alpha, self.n, self.ksat = P(0.01), P(1.5), P(0.4)
        self.ponded_depth_max = torch.tensor(0.0, dtype=torch.float64)
        self.ending_volume = torch.tensor(50.0, dtype=torch.float64)
        self.resets = 0

    def set_internal_states(self):
        self.resets += 1

    def forward_record(self, x, outputs=("runoff",), on_status="raise"):
        x = torch.as_tensor(x, dtype=torch.float64)
        if x.dim() == 2:
            x = x[None]
        p = x[..., 0].transpose(0, 1)  # [T, sites]
        runoff = p * self.ksat[0] * self.alpha[0] * 100.0 + self.n[1] * 0.01 * p ** 2
        out = {k: torch.zeros_like(runoff) for k in outputs}
        out["runoff"] = runoff
        out["precip"] = p
        out["ending_volume"] = 50.0 + torch.cumsum(p - runoff.detach(), dim=0)
        out["start_volume"] = torch.full((p.shape[1],), 50.0, dtype=torch.float64)
        out["status"] = torch.zeros(p.shape[1], dtype=torch.int32)
        if p.shape[1] == 1:
            out = {k: (v[:, 0] if v.dim() == 2 else v) for k, v in out.items()}
        return out


def test_derive_time_config_matches_reference_arithmetic():
    c = A.derive_time_config(_cfg(endtime=7500.0, subcycle=300.0))
    m = c["models"]
    assert m["num_subcycles"] == 12 and m["nsteps"] == 7500 and m["subcycle_length_h"] == 300.0 * (1 / 3600.0)
    c = A.derive_time_config(_cfg(endtime=3000.0, subcycle=3600.0))
    assert c["models"]["num_subcycles"] == 1 and c["models"]["nsteps"] == 3000
    ns = SimpleNamespace(conversions=SimpleNamespace(hr_to_sec=3600.0),
                         models=SimpleNamespace(endtime=10.0, subcycle_length=300.0, forcing_resolution=300.0))
    A.derive_time_config(ns)  # synthetic 5-minute forcing (SURVEY C2)
    assert ns.models.num_subcycles == 1 and ns.models.nsteps == 120


def test_losses_and_nse():
    torch.set_default_dtype(torch.float64)
    rb = A.RangeBoundLoss(LB, UB)
    mk = lambda vals: torch.nn.ParameterList([torch.nn.Parameter(torch.tensor(v, dtype=torch.float64)) for v in vals])
    alpha, n, ks, pdm = mk([0.02, 0.001, 0.01]), mk([0.9, 5.5, 2.0]), mk([31.0, 0.5, 1e-7]), torch.tensor(11.0)
    got = float(rb([alpha, n, ks, pdm]))
    # by hand (sum over the upper violations, MEAN over the lower ones, sic): loss.py:22-30
    want = (0.02 - 0.015) + (0.0015 - 0.001) / 3 + (5.5 - 5.0) + (1.0 - 0.9) / 3 + (31.0 - 30) + (1e-6 - 1e-7) / 3 + 1.0
    assert got == pytest.approx(want, rel=1e-14)
    assert float(rb([mk([0.01] * 3), mk([1.5] * 3), mk([1.0] * 3), torch.tensor(0.0)])) == 0.0
    y, t = torch.tensor([0.1, 0.4, 0.2]), torch.tensor([0.0, 0.5, 0.1])
    assert float(A.mse_loss(y, t)) == pytest.approx(0.01)
    assert A.calculate_nse(y.numpy(), t.numpy()) == pytest.approx(1 - 0.03 / float(((t - t.mean()) ** 2).sum()))


def test_reference_observations_are_the_seeded_series():
    torch.set_default_dtype(torch.float64)
    torch.manual_seed(0)
    want = torch.rand([17])  # data/Data.py:40 right after the agent's manual_seed(0)
    assert torch.equal(A.reference_observations(17), want)


def test_mass_balance_report():
    lines = []
    tot = dict(precip=10.0, runoff=1.5, AET=2.0, ponded_water=0.25, percolation=0.0, ending_volume=56.25, infiltration=8.0,
               giuh_runoff=1.4, PET=3.0, discharge=1.4)
    err = A.mass_balance_report(tot, 50.0, giuh_queue_sum=0.1, emit=lines.append)
    assert err == pytest.approx(0.0, abs=1e-12)
    assert any("GIUH runoff" in l and "1.500000" in l for l in lines) and "Global balance" in lines[-1]


def test_train_checkpoint_roundtrip(tmp_path):
    rng = np.random.default_rng(3)
    x = np.abs(rng.normal(size=(48, 2))) * 0.3
    ag = A.DifferentiableLGAR(_cfg(), model=ToyModel(), x=x)
    assert ag.x.shape == (1, 48, 2) and ag.y.shape == (1, 48)
    ag.train()
    assert ag.current_epoch == 2 and ag.model.resets == 2 and len(ag.history) == 2
    assert ag.history[1][1] < ag.history[0][1]  # the loss went down
    assert abs(ag.last_balance_error) < 1e-9
    ck = str(tmp_path / "ck.pth.tar")
    ag.save_checkpoint(ck, is_best=1)
    assert os.path.exists(tmp_path / "model_best.pth.tar")
    ag2 = A.DifferentiableLGAR(_cfg(), model=ToyModel(), x=x)
    ag2.load_checkpoint(ck)
    assert ag2.current_epoch == 2
    for p, q in zip(ag.model.parameters(), ag2.model.parameters()):
        assert torch.equal(p, q)
    ag.train_one_epoch(); ag2.train_one_epoch()  # same Adam state -> same next step
    for p, q in zip(ag.model.parameters(), ag2.model.parameters()):
        assert torch.equal(p, q)


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    rng = np.random.default_rng(5)
    x = np.abs(rng.normal(size=(2, 48, 2))) * 0.3  # two sites: one per rank
    y = np.abs(rng.normal(size=(2, 48))) * 0.05
    ag = A.DifferentiableLGAR(_cfg(epochs=1), model=ToyModel(), x=x[rank], y=y[rank])
    ag.train()
    out[rank] = [p.detach().numpy().copy() for p in ag.model.parameters()] + [ag.history[0][1]]
    dist.destroy_process_group()


def test_two_ranks_equal_two_sites_in_one_process():
    port = 31000 + os.getpid() % 2000
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    rng = np.random.default_rng(5)
    x = np.abs(rng.normal(size=(2, 48, 2))) * 0.3
    y = np.abs(rng.normal(size=(2, 48))) * 0.05
    ag = A.DifferentiableLGAR(_cfg(epochs=1), model=ToyModel(), x=x, y=y)  # both sites, one process
    ag.train()
    want = [p.detach().numpy() for p in ag.model.parameters()]
    for r in range(2):
        for got, w in zip(out[r][:-1], want):
            np.testing.assert_allclose(got, w, rtol=1e-12, atol=1e-15)
        assert out[r][-1] == pytest.approx(ag.history[0][1], rel=1e-12)
