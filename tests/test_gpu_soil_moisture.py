"""-m gpu: the soil-moisture outputs (include/lgar_b200.h): theta at sensor depths and the water of every layer after
each forcing step, from both kernels and through autograd.

* against the Python reference's own front lists (the forward goldens) and against the kernel's dumped fronts;
* sum of the layer waters = ENDING_VOLUME bit for bit; nothing else changes when the outputs are requested;
* windows, pipelined windows and placement do not change them;
* gradients: layer water against ending volume, and reverse mode against the CPU oracle's forward-mode tangents."""
import math
import os

import numpy as np
import pytest
import torch

from conftest import golden_names, load_golden, max_excess
from oracle_moisture import moisture_batch
from soil_moisture_ref import counts_from_layers, layer_water, outputs_of_dump, theta_at

pytestmark = pytest.mark.gpu

GOLDEN_DEPTHS = (1.0, 5.0, 10.0, 20.0, 43.9, 44.0, 44.1, 50.0, 100.0, 175.0, 199.9, 200.0)
SENSORS = (5.0, 10.0, 20.0, 50.0, 100.0)
FORWARD_GOLDENS = [nm for nm in golden_names() if "fronts" in load_golden(nm).files]


def _bits(x):
    return x.contiguous().view(torch.int64)


def _bench_like(B=2048, T=300, sites=4, rank=3, **kw):
    from lgar_b200 import workloads, ColumnEnsemble
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=sites, rank=rank)
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, **kw)
    return we, ens


@pytest.mark.parametrize("name", FORWARD_GOLDENS)
def test_against_reference_front_lists(name):
    """W_l and theta(z) of the kernel against the same quantities derived from the reference's front lists after
    every step (list membership from the golden's layer_num, which must group the list: the test asserts it)."""
    from gpu_common import ensemble_from_golden
    from lgar_b200 import forward_raw
    g = load_golden(name)
    T = g["forcing"].shape[0]
    cs = int(g["crash_step"])
    n_ok = T if cs < 0 else cs
    thick = [float(x) for x in g["layer_thickness"]]
    W_ref, th_ref = outputs_of_dump(g["fronts"][:n_ok], g["front_layer"][:n_ok], g["nfronts"][:n_ok], thick,
                                    GOLDEN_DEPTHS)
    th_got = []
    for part in (GOLDEN_DEPTHS[:6], GOLDEN_DEPTHS[6:]):
        ens, a, n, k = ensemble_from_golden(g, copies=1, moisture_depths=part)
        res, _ = forward_raw(ens, a, n, k, outputs=("ending_volume",), moisture=True, layer_water=True)
        th_got.append(res.moisture[:, :, 0].T.cpu().numpy())
        W_got = res.layer_water[:, :, 0].T.cpu().numpy()   # [T, L]
        if n_ok < T:   # crashed columns: NaN from the crash step on
            assert np.isnan(W_got[n_ok:]).all() and np.isnan(th_got[-1][n_ok:]).all()
    th_got = np.concatenate(th_got, axis=1)[:n_ok]
    W_got = W_got[:n_ok]
    ex = max_excess(W_got, W_ref)
    assert ex <= 1.0, f"layer water exceeds 1e-9 rel + 1e-12 cm by factor {ex:.3g}"
    ex = max_excess(th_got, th_ref)
    assert ex <= 1.0, f"theta(z) exceeds 1e-9 rel + 1e-12 by factor {ex:.3g}"
    inside = np.array(GOLDEN_DEPTHS) <= sum(thick)
    assert not np.isnan(th_got[:, inside]).any(), "a depth inside the column found no front"
    assert np.isnan(th_got[:, ~inside]).all()


def test_against_the_kernels_own_fronts_bit_for_bit():
    """One dump_fronts run: both outputs equal the restatement on the dumped front lists, every bit."""
    from lgar_b200 import ColumnEnsemble, forward_raw, workloads
    g = load_golden("phil_4500_600")
    B, T = 64, 300
    rng = np.random.default_rng(7)
    a, n, k = workloads.sample_parameters(rng, B)
    rep = lambda v: np.repeat(np.asarray(v, dtype=np.float64).reshape(3, 1), B, axis=1)
    depths = (1.0, 10.0, 43.9, 44.0, 44.1, 100.0, 175.0, 200.0)
    ens = ColumnEnsemble(theta_r=rep(g["theta_r"]), theta_e=rep(g["theta_e"]), thickness=rep(g["layer_thickness"]),
                         forcing=g["forcing"][:T], moisture_depths=depths)
    res, _ = forward_raw(ens, a, n, k, outputs=("ending_volume",), dump_fronts=True, moisture=True, layer_water=True)
    torch.cuda.synchronize()
    fr, fl, nf = res.fronts.cpu().numpy(), res.front_layer.cpu().numpy(), res.num_fronts.cpu().numpy()
    th, W = res.moisture.cpu().numpy(), res.layer_water.cpu().numpy()
    st, cs = res.status.cpu().numpy(), res.crash_step.cpu().numpy()
    thick = [float(x) for x in g["layer_thickness"]]
    checked = 0
    for b in range(B):
        n_ok = T if st[b] == 0 else cs[b]
        for t in range(n_ok):
            cnt = counts_from_layers(fl[t, :, b], int(nf[t, b]), 3)
            d, q = fr[t, :nf[t, b], 0, b], fr[t, :nf[t, b], 1, b]
            ref_w = np.array(layer_water(d, q, cnt, thick))
            ref_t = np.array([theta_at(z, d, q, cnt, thick) for z in depths])
            assert np.array_equal(W[:, t, b].view(np.int64), ref_w.view(np.int64)), (b, t, W[:, t, b], ref_w)
            assert np.array_equal(th[:, t, b].view(np.int64), ref_t.view(np.int64)), (b, t, th[:, t, b], ref_t)
            checked += 1
        assert np.isnan(W[:, n_ok:, b]).all() and np.isnan(th[:, n_ok:, b]).all()
    assert checked >= B * T // 2


def test_layer_water_sums_to_ending_volume_bit_for_bit():
    from lgar_b200 import forward_raw
    we, ens = _bench_like(moisture_depths=SENSORS)
    res, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=("ending_volume",), layer_water=True)
    W = res.layer_water
    total = W[0] + (W[1] + W[2])
    ok = res.status == 0
    assert int(ok.sum()) > 1000
    assert torch.equal(_bits(total[:, ok]), _bits(res["ending_volume"][:, ok]))


def test_nothing_else_changes():
    """Requesting the soil-moisture outputs leaves every other output bit-identical, with and without checkpoints;
    with their gradients not requested, the reverse pass gives bit-identical parameter gradients."""
    from lgar_b200 import forward_raw, lgar_columns, OUT_NAMES
    we, ens = _bench_like(B=3000, T=240, moisture_depths=SENSORS)
    for keep in (False, True):
        ref, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUT_NAMES, num_fronts=True, keep_checkpoints=keep)
        new, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUT_NAMES, num_fronts=True, keep_checkpoints=keep,
                             moisture=True, layer_water=True)
        for x, y in ((ref.per_step, new.per_step), (ref.sums, new.sums), (ref.start_volume, new.start_volume)):
            assert torch.equal(_bits(x), _bits(y))
        for x, y in ((ref.status, new.status), (ref.crash_step, new.crash_step), (ref.num_fronts, new.num_fronts)):
            assert torch.equal(x, y)
    grads = []
    for extra in ((), ("moisture", "layer_water")):
        mk = lambda v: torch.tensor(v, device="cuda", requires_grad=True)
        A, N, K = mk(we.alpha), mk(we.n), mk(we.ksat)
        out = lgar_columns(A, N, K, ens, outputs=("runoff", "AET", "ending_volume") + extra)
        ok = out["status"] == 0
        loss = (torch.nan_to_num(out["runoff"] + out["AET"]).sum(0) + out["sums"][4])[ok].sum()
        loss.backward()
        grads.append((A.grad, N.grad, K.grad))
    for x, y in zip(*grads):
        assert torch.equal(_bits(x), _bits(y))


def test_pipelined_windows_equal_one_launch():
    from lgar_b200 import forward_raw
    import bench
    we, ens = _bench_like(B=40_000, T=200, sites=8, rank=2, moisture_depths=SENSORS)
    T = ens.num_steps
    full, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=("runoff",), moisture=True, layer_water=True)
    res, ws = None, None
    for i, (t0, t1) in enumerate(bench.segments(T, 20)):
        res, ws = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=("runoff",), workspace=ws, window=(t0, t1), into=res,
                              pipeline_seq=i + 1, moisture=True, layer_water=True)
    torch.cuda.synchronize()
    assert (full.status != 0).any()
    assert torch.equal(_bits(res.moisture), _bits(full.moisture))
    assert torch.equal(_bits(res.layer_water), _bits(full.layer_water))
    assert torch.equal(_bits(res.per_step), _bits(full.per_step))


def _mse_loss(out, ok, obs_theta=0.3, obs_water=20.0):
    th = out["moisture"][:, :, ok]
    W = out["layer_water"][:, :, ok]
    return ((th - obs_theta) ** 2).sum() + ((W - obs_water) ** 2).sum() * 1e-3


def test_placement_changes_neither_values_nor_gradients():
    from lgar_b200 import lgar_columns
    res = []
    for balanced in (False, True):
        we, ens = _bench_like(B=3000, T=200, sites=6, rank=2, moisture_depths=SENSORS)
        if balanced:
            ens.balance(we.ksat)
        mk = lambda v: torch.tensor(v, device="cuda", requires_grad=True)
        A, N, K = mk(we.alpha), mk(we.n), mk(we.ksat)
        out = lgar_columns(A, N, K, ens, outputs=("moisture", "layer_water"))
        ok = out["status"] == 0
        _mse_loss(out, ok).backward()
        res.append((out["moisture"].detach(), out["layer_water"].detach(), A.grad, N.grad, K.grad, ok))
    ok = res[0][5]
    assert torch.equal(ok, res[1][5])
    for x, y in zip(res[0][:2], res[1][:2]):
        assert torch.equal(_bits(x), _bits(y))
    for x, y in zip(res[0][2:5], res[1][2:5]):
        assert torch.equal(_bits(x[:, ok]), _bits(y[:, ok]))


def test_layer_water_gradient_equals_ending_volume_gradient():
    """sum_t W_0 + (W_1 + W_2) is sum_t ENDING_VOLUME: the two losses give the same dL/d(alpha, n, ksat, ponded_depth_max)."""
    from lgar_b200 import lgar_columns
    we, ens = _bench_like(B=512, T=300, sites=2, rank=5, ponded_depth_max=0.5)
    got = []
    for via in ("layer_water", "ending_volume"):
        mk = lambda v: torch.tensor(v, device="cuda", requires_grad=True)
        A, N, K = mk(we.alpha), mk(we.n), mk(we.ksat)
        P = torch.full((512,), 0.5, dtype=torch.float64, device="cuda", requires_grad=True)
        out = lgar_columns(A, N, K, ens, outputs=(via,), ponded_depth_max=P)
        ok = out["status"] == 0
        if via == "layer_water":
            W = out["layer_water"]
            loss = (W[0] + (W[1] + W[2]))[:, ok].sum()
        else:
            loss = out["ending_volume"][:, ok].sum()
        loss.backward()
        got.append([A.grad[:, ok], N.grad[:, ok], K.grad[:, ok], P.grad[ok]])
    assert int(ok.sum()) > 400
    for x, y in zip(*got):
        scale = y.abs().max()
        assert bool(((x - y).abs() <= 1e-12 * y.abs() + 1e-12 * scale).all()), float((x - y).abs().max() / scale)


def _oracle_grads(cfgs, forcing, site, depths, okn, obs_theta=0.3, obs_water=20.0, chunk=16):
    """d(_mse_loss)/d(alpha, n, ksat) per column from the oracle's forward-mode tangents: [B, 3, L]."""
    B = len(cfgs)
    out = np.zeros((B, 3, 3))
    for lo in range(0, B, chunk):
        idx = [b for b in range(lo, min(B, lo + chunk))]
        r = moisture_batch([cfgs[b] for b in idx], forcing, depths, site=None if site is None else site[idx],
                           nthreads=16, tangents=True)
        for j, b in enumerate(idx):
            if not okn[b]:
                continue
            assert r["status"][j] == 0
            th, dth = r["moisture"][j], r["dmoisture"][j]          # [T,D], [T,D,9]
            W, dW = r["layer_water"][j], r["dlayer_water"][j]      # [T,L], [T,L,9]
            g = (2.0 * (th - obs_theta))[:, :, None] * dth
            g = g.sum((0, 1)) + ((2.0 * (W - obs_water))[:, :, None] * dW).sum((0, 1)) * 1e-3
            out[b] = g.reshape(3, 3)
    return out


def test_gradients_match_oracle_tangents_on_random_members():
    from lgar_b200 import ColumnEnsemble, lgar_columns, workloads
    from oracle import lgar_oracle as O
    g = load_golden("phil_4500_600")
    T, B = 200, 32
    forcing = g["forcing"][40:40 + T]
    rng = np.random.default_rng(11)
    a, n, k = workloads.sample_parameters(rng, B)
    rep = lambda v: np.repeat(np.asarray(v, dtype=np.float64).reshape(3, 1), B, axis=1)
    ens = ColumnEnsemble(theta_r=rep(g["theta_r"]), theta_e=rep(g["theta_e"]), thickness=rep(g["layer_thickness"]),
                         forcing=forcing, chunk_steps=48, moisture_depths=SENSORS)
    mk = lambda v: torch.tensor(v, device="cuda", requires_grad=True)
    A, N, K = mk(a), mk(n), mk(k)
    out = lgar_columns(A, N, K, ens, outputs=("moisture", "layer_water"))
    ok = out["status"] == 0
    _mse_loss(out, ok).backward()
    got = np.stack([A.grad.cpu().numpy(), N.grad.cpu().numpy(), K.grad.cpu().numpy()])   # [3, L, B]
    okn = ok.cpu().numpy()
    cfgs = [O.make_cfg(a[:, b], n[:, b], k[:, b], g["theta_r"], g["theta_e"]) for b in range(B)]
    ref = _oracle_grads(cfgs, forcing, None, SENSORS, okn)
    assert okn.sum() >= 20
    for b in np.nonzero(okn)[0]:
        scale = max(np.abs(ref[b]).max(), 1e-300)
        np.testing.assert_allclose(got[:, :, b], ref[b], rtol=1e-8, atol=1e-10 * scale, err_msg=f"column {b}")


def test_full_year_gradients_match_oracle_tangents():
    from lgar_b200 import lgar_columns
    from oracle import lgar_oracle as O
    B, T = 64, 8760
    we, ens = _bench_like(B=B, T=T, sites=2, rank=4, moisture_depths=SENSORS)
    mk = lambda v: torch.tensor(v, device="cuda", requires_grad=True)
    A, N, K = mk(we.alpha), mk(we.n), mk(we.ksat)
    out = lgar_columns(A, N, K, ens, outputs=("moisture", "layer_water"))
    ok = out["status"] == 0
    _mse_loss(out, ok).backward()
    assert ens.check_tape_overflow() == 0
    got = np.stack([A.grad.cpu().numpy(), N.grad.cpu().numpy(), K.grad.cpu().numpy()])
    okn = ok.cpu().numpy()
    assert okn.sum() >= 30
    cfgs = [O.make_cfg(we.alpha[:, b], we.n[:, b], we.ksat[:, b], we.theta_r[:, b], we.theta_e[:, b],
                       iter_cap=1_000_000) for b in range(B)]
    ref = _oracle_grads(cfgs, we.forcing, we.site_index, SENSORS, okn)
    worst = 0.0
    for b in np.nonzero(okn)[0]:
        scale = max(np.abs(ref[b]).max(), 1e-300)
        err = np.abs(got[:, :, b] - ref[b]) / (1e-8 * np.abs(ref[b]) + 1e-10 * scale)
        worst = max(worst, float(err.max()))
    assert worst <= 1.0, f"full-year gradients exceed 1e-8 rel + 1e-10 x max|grad| by factor {worst:.3g}"


def test_values_bit_exact_against_same_pow_oracle_full_year():
    """256 full-year columns of the C4 shard: with the CUDA path's pow on both sides the two outputs agree bit for bit."""
    from lgar_b200 import ColumnEnsemble, forward_raw, workloads
    from oracle import lgar_oracle as O
    B, T = 256, 8760
    big = workloads.synthetic_sites_ensemble(B=125_000, T=T)
    cols = np.linspace(0, 124_999, B).astype(np.int64)
    sl = lambda x: np.ascontiguousarray(x[:, cols])
    ens = ColumnEnsemble(theta_r=sl(big.theta_r), theta_e=sl(big.theta_e), thickness=sl(big.thickness),
                         forcing=big.forcing, site_index=big.site_index[cols], moisture_depths=SENSORS)
    res, _ = forward_raw(ens, sl(big.alpha), sl(big.n), sl(big.ksat), outputs=(), per_step=False, moisture=True,
                         layer_water=True)
    torch.cuda.synchronize()
    st = res.status.cpu().numpy()
    th, W = res.moisture.cpu().numpy(), res.layer_water.cpu().numpy()
    cfgs = [O.make_cfg(big.alpha[:, b], big.n[:, b], big.ksat[:, b], big.theta_r[:, b], big.theta_e[:, b],
                       thickness=big.thickness[:, b], iter_cap=1_000_000) for b in cols]
    r = moisture_batch(cfgs, big.forcing, SENSORS, site=big.site_index[cols], nthreads=min(32, os.cpu_count() or 1),
                       variant="devpow")
    ITER_CAP = 7
    use = (st == r["status"]) & (st == 0)
    assert int(((st == ITER_CAP) | (r["status"] == ITER_CAP)).sum()) <= B // 20
    assert int(use.sum()) >= B // 2
    for j in np.nonzero(use)[0]:
        assert np.array_equal(W[:, :, j].T.view(np.int64), r["layer_water"][j].view(np.int64)), f"column {cols[j]}"
        assert np.array_equal(th[:, :, j].T.view(np.int64), r["moisture"][j].view(np.int64)), f"column {cols[j]}"


def test_shared_parameters_reduce_in_library_and_model_surface():
    """[L] (shared) parameters: the in-library reduced sum equals the sum of the per-column gradients; the dpLGAR module
    returns the outputs from forward_record and its one-row forward reproduces them row by row."""
    from lgar_b200 import lgar_columns, workloads, ColumnEnsemble, dpLGAR
    B, T = 1500, 240
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=3, rank=5)
    col = 7
    for x in (we.alpha, we.n, we.ksat):
        x[:] = x[:, col:col + 1]
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, moisture_depths=SENSORS)
    grads = []
    for shared in (False, True):
        mk = lambda v: torch.tensor(np.ascontiguousarray(v[:, col]) if shared else v, device="cuda", requires_grad=True)
        A, N, K = mk(we.alpha), mk(we.n), mk(we.ksat)
        out = lgar_columns(A, N, K, ens, outputs=("moisture", "layer_water"))
        ok = out["status"] == 0
        assert int(ok.sum()) == B
        (_mse_loss(out, ok) + out["layer_theta"].sum()).backward()
        grads.append((A.grad, N.grad, K.grad))
    for per_col, shared in zip(*grads):
        assert shared.shape == (3,)
        assert bool(((shared - per_col.sum(1)).abs() <= 1e-12 * per_col.abs().sum(1) + 1e-300).all())

    g = load_golden("phil_4500_400_pdm2")
    cfg = dict(constants=dict(frozen_factor=float(g["frozen_factor"]), nint=int(g["nint"])),
               data=dict(layer_soil_type=[12, 13, 14], layer_thickness=[float(x) for x in g["layer_thickness"]],
                         initial_psi=float(g["initial_psi"]), ponded_depth_max=float(g["ponded_depth_max"]),
                         wilting_point_psi=float(g["wilting_point_psi"]),
                         giuh_ordinates=[float(x) for x in g["giuh_ordinates"]], moisture_depths=[5.0, 44.0, 120.0]),
               models=dict(subcycle_length_h=float(g["subcycle_length_h"]), num_subcycles=int(g["num_subcycles"])))
    model = dpLGAR(cfg, theta_r=g["theta_r"], theta_e=g["theta_e"])
    assert model.moisture_depths == (5.0, 44.0, 120.0)
    assert dpLGAR(cfg, theta_r=g["theta_r"], theta_e=g["theta_e"], moisture_depths=[10.0]).moisture_depths == (10.0,)
    T = 60
    x = torch.tensor(g["forcing"][:T])
    rec = model.forward_record(x)
    assert rec["moisture"].shape == (T, 3) and rec["layer_water"].shape == (T, 3) and rec["layer_theta"].shape == (T, 3)
    rec["moisture"].sum().backward()
    assert all(math.isfinite(float(p.grad)) for p in model.alpha)
    for t in range(T):
        model(x[t])
        for k in ("precip", "PET", "AET", "infiltration", "runoff", "percolation", "giuh_runoff", "discharge"):
            setattr(model, k, torch.tensor(0.0, dtype=torch.float64))
        assert torch.equal(model.soil_moisture, rec["moisture"][t].detach().cpu()), t
        assert torch.equal(model.layer_water, rec["layer_water"][t].detach().cpu()), t
