"""-m gpu: ensemble-scale checks of the CUDA path (through the C ABI).

* against the CPU oracle on a random parameter ensemble (status of every column identical, sums within tolerance);
* size-independent properties at the bench's column count (BASELINE.json C4 shard, shortened record): the global
  mass balance of every OK column closes, two launches give identical bits, the result of a column does not depend
  on which tile / lane / shard it runs in, nor on the chunk length of the scheduler, and a record split in two
  `resume` launches equals one launch;
* ragged shapes: one column, one step, column counts that are not a multiple of 32, records that are not a multiple
  of the chunk length."""
import numpy as np
import pytest
import torch

from conftest import max_excess

pytestmark = pytest.mark.gpu
OUTS = ("runoff", "percolation", "AET", "infiltration", "ending_volume", "ponded_water", "giuh_runoff", "precip", "PET",
        "discharge")


def _ens(we, cols=None, T=None, **kw):
    from lgar_b200 import ColumnEnsemble
    sl = slice(None) if cols is None else cols
    f = we.forcing if T is None else we.forcing[:, :T]
    return ColumnEnsemble(theta_r=np.ascontiguousarray(we.theta_r[:, sl]), theta_e=np.ascontiguousarray(we.theta_e[:, sl]),
                          thickness=np.ascontiguousarray(we.thickness[:, sl]), forcing=np.ascontiguousarray(f),
                          site_index=np.ascontiguousarray(we.site_index[sl]), **kw)


def _run(we, cols=None, T=None, outputs=("runoff", "AET"), **kw):
    from lgar_b200 import forward_raw
    sl = slice(None) if cols is None else cols
    ens = _ens(we, cols, T, **kw)
    res, ws = forward_raw(ens, np.ascontiguousarray(we.alpha[:, sl]), np.ascontiguousarray(we.n[:, sl]),
                          np.ascontiguousarray(we.ksat[:, sl]), outputs=outputs)
    torch.cuda.synchronize()
    return res, ws, ens


def test_random_ensemble_matches_oracle():
    from lgar_b200 import workloads
    from oracle import lgar_oracle as O
    B, T = 1536, 400
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=8, rank=3)
    res, _, _ = _run(we, outputs=OUTS)
    sums = res.sums.cpu().numpy()      # [NOUT, B]
    status = res.status.cpu().numpy()
    worst = 0.0
    for s in range(8):
        idx = np.nonzero(we.site_index == s)[0]
        cfgs = [O.make_cfg(we.alpha[:, b], we.n[:, b], we.ksat[:, b], we.theta_r[:, b], we.theta_e[:, b],
                           thickness=we.thickness[:, b]) for b in idx]
        osums, ost = O.forward_batch(cfgs, we.forcing[s], nthreads=16)
        np.testing.assert_array_equal(status[idx], ost)  # the same columns fail, with the same status
        ok = ost == 0
        for k, name in enumerate(OUTS):
            worst = max(worst, max_excess(sums[k, idx[ok]], osums[ok, k], rtol=1e-9, atol=1e-10))
    assert worst <= 1.0, f"CUDA vs oracle sums exceed 1e-9 rel by factor {worst:.3g}"
    assert (status == 0).sum() > 0.9 * B


def test_properties_at_bench_width():
    from lgar_b200 import workloads, forward_raw
    B, T = 125_000, 192
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=128, rank=0)
    res, ws, ens = _run(we, outputs=OUTS)
    st = res.status.cpu().numpy()
    ok = st == 0
    assert ok.mean() > 0.95
    s = {name: res.sums[k].cpu().numpy() for k, name in enumerate(OUTS)}
    start = res.start_volume.cpu().numpy()
    # MassBalance.report_mass (physics/MassBalance.py:84-92): the global balance of every surviving column closes
    err = start + s["precip"] - s["runoff"] - s["AET"] - s["ponded_water"] - s["percolation"] - s["ending_volume"]
    closes = np.abs(err) < 1e-7
    assert closes[ok].mean() > 0.98, f"only {closes[ok].mean():.4f} of the OK columns close the global mass balance"
    assert np.median(np.abs(err[ok])) < 1e-9
    # the remaining columns do not conserve mass in the REFERENCE either (e.g. the bottom flux dropped in the
    # surficial-front branch, Q7, or water leaving through wetting_front_cross_domain_boundary): same error in the oracle
    from oracle import lgar_oracle as O
    bad = np.nonzero(ok & ~closes)[0][:8]
    for b in bad:
        cfg = O.make_cfg(we.alpha[:, b], we.n[:, b], we.ksat[:, b], we.theta_r[:, b], we.theta_e[:, b], thickness=we.thickness[:, b])
        r = O.forward(cfg, we.forcing[we.site_index[b]], fronts=False)
        assert r["status"] == 0
        oerr = (start[b] + r["precip"].sum() - r["runoff"].sum() - r["AET"].sum() - r["ponded_water"][-1]
                - r["percolation"].sum() - r["ending_volume"][-1])
        assert abs(oerr - err[b]) < 1e-8, (b, oerr, err[b])
    # per-step series are consistent with the sums; runoff and precipitation are non-negative (AET is not: the
    # dry-over-wet correction subtracts its mass change from it, models/dpLGAR.py:364-366); AET never exceeds PET
    for name in ("runoff", "AET", "infiltration", "precip"):
        series = res[name].cpu().numpy()[:, ok]
        if name in ("runoff", "precip"):
            assert (series >= 0).all(), name
        np.testing.assert_allclose(series.sum(axis=0), s[name][ok], rtol=1e-12, atol=1e-13)
    assert (res["AET"].cpu().numpy()[:, ok] <= res["PET"].cpu().numpy()[:, ok] + 1e-15).all()
    # determinism: a second launch into the same workspace gives identical bits
    res2, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUTS, workspace=ws)
    torch.cuda.synchronize()
    assert torch.equal(res.sums.view(torch.int64), res2.sums.view(torch.int64))
    assert torch.equal(res.status, res2.status) and torch.equal(res.crash_step, res2.crash_step)
    # placement invariance: a shard of the columns (other tiles, other lanes: offset not a multiple of 32) and a
    # different chunk length give the same bits for every column
    lo, hi = 40_013, 40_013 + 9_999
    part, _, _ = _run(we, cols=slice(lo, hi), outputs=OUTS, chunk_steps=48)
    assert torch.equal(part.sums.view(torch.int64), res.sums[:, lo:hi].contiguous().view(torch.int64))
    assert torch.equal(part.status, res.status[lo:hi])


def test_resume_equals_one_launch():
    from lgar_b200 import workloads, forward_raw
    B, T, T1 = 4097, 160, 70
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=4, rank=1)
    full, _, _ = _run(we)
    first_ens = _ens(we, T=T1)
    r1, ws = forward_raw(first_ens, we.alpha, we.n, we.ksat, outputs=("runoff", "AET"))
    from lgar_b200 import ColumnEnsemble
    second = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness,
                            forcing=np.ascontiguousarray(we.forcing[:, T1:]), site_index=we.site_index, resume=True)
    r2, _ = forward_raw(second, we.alpha, we.n, we.ksat, outputs=("runoff", "AET"), workspace=ws)
    torch.cuda.synchronize()
    ok = (full.status == 0)
    got = torch.cat([r1["runoff"], r2["runoff"]])[:, ok]
    assert torch.equal(got.contiguous().view(torch.int64), full["runoff"][:, ok].contiguous().view(torch.int64))
    got = torch.cat([r1["AET"], r2["AET"]])[:, ok]
    assert torch.equal(got.contiguous().view(torch.int64), full["AET"][:, ok].contiguous().view(torch.int64))


@pytest.mark.parametrize("B,T", [(1, 1), (1, 97), (31, 64), (33, 65), (1000, 3)])
def test_ragged_shapes(B, T):
    from lgar_b200 import workloads
    big = workloads.synthetic_sites_ensemble(B=1024, T=128, sites=2, rank=2)
    ref, _, _ = _run(big, outputs=OUTS)
    cols = slice(500, 500 + B) if B < 1000 else slice(0, 1000)
    part, _, _ = _run(big, cols=cols, T=T, outputs=OUTS)
    ok = (part.status == 0).cpu().numpy()
    a = part["runoff"].cpu().numpy()[:, ok]
    b = ref["runoff"].cpu().numpy()[:T, cols][:, ok]
    np.testing.assert_array_equal(a, b)
    a = part["ending_volume"].cpu().numpy()[:, ok]
    b = ref["ending_volume"].cpu().numpy()[:T, cols][:, ok]
    np.testing.assert_array_equal(a, b)


def test_front_overflow_fallback():
    """Columns that overflow the front list are rerun with the 32-front instantiation: with an 8-front base kernel
    plus the fallback every column must give the bits of the 16-front kernel."""
    from lgar_b200 import workloads, forward_raw
    B, T = 16384, 640
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=16, rank=0)
    ref, _, _ = _run(we, outputs=OUTS)                                   # 16 fronts
    small, _, _ = _run(we, outputs=OUTS, max_fronts=8)                   # 8 fronts, no fallback
    n_over = int((small.status == 6).sum())
    assert n_over > 0, "the case must contain overflowing columns"
    ens8 = _ens(we, max_fronts=8)
    fb, _ = forward_raw(ens8, we.alpha, we.n, we.ksat, outputs=OUTS, overflow_fallback=True)
    torch.cuda.synchronize()
    assert fb.overflow_reruns == n_over
    assert torch.equal(fb.status, ref.status) and torch.equal(fb.crash_step, ref.crash_step)
    ok = ref.status == 0
    assert torch.equal(fb.sums[:, ok].contiguous().view(torch.int64), ref.sums[:, ok].contiguous().view(torch.int64))
    assert torch.equal(fb["runoff"][:, ok].contiguous().view(torch.int64), ref["runoff"][:, ok].contiguous().view(torch.int64))


def test_subset_carries_every_field():
    """ColumnEnsemble.subset (the 32-front rerun's sub-ensemble): per-column fields are those of the indexed columns,
    the forcing is shared, the placement, resume and the last backward pass's results are not carried, every other
    field equals the parent's.  A field added to ColumnEnsemble that subset does not handle fails here."""
    import dataclasses
    from lgar_b200 import workloads
    B = 100
    we = workloads.synthetic_sites_ensemble(B=B, T=20, sites=3, rank=0)
    ens = _ens(we, initial_psi=np.linspace(1000.0, 3000.0, B), ponded_depth_max=0.5, moisture_depths=(5.0, 30.0),
               nint=60, iter_cap=12345, use_closed_form_G=True, reverse_counters=True, resume=True)
    ens.balance(we.ksat)
    ens.last_tape_overflow = torch.zeros(B, dtype=torch.int32, device="cuda")
    idx = torch.tensor([3, 17, 64, 99], device="cuda")
    sub = ens.subset(idx, max_fronts=32)
    default = {f.name: (f.default_factory() if f.default_factory is not dataclasses.MISSING else f.default)
               for f in dataclasses.fields(ens)}
    for f in dataclasses.fields(ens):
        got, parent = getattr(sub, f.name), getattr(ens, f.name)
        if f.name in ("column_order", "resume", "_keep") or f.name.startswith("last_"):
            assert not isinstance(got, torch.Tensor) and got == default[f.name], f.name
        elif f.name == "max_fronts":
            assert got == 32
        elif f.name == "forcing":
            assert got.data_ptr() == parent.data_ptr()
        elif isinstance(parent, torch.Tensor) and parent.shape[-1:] == (B,):
            assert torch.equal(got, parent[..., idx]), f.name
        elif isinstance(parent, torch.Tensor):
            assert torch.equal(got, parent), f.name
        else:
            assert got == parent, f.name
    assert sub.num_columns == 4 and sub.num_layers == ens.num_layers


def test_flat_column_mass_run_ends_with_iter_cap_quickly():
    """A column whose free-drainage front has the theta of the front below it: the column mass does not depend on the
    depth check_column_mass steps (Layer.py:681-701), the reference never leaves that loop, this library answers with
    the capacity status ITER_CAP -- at the step where the oracle's literal loop passes 1e6 iterations, and WITHOUT
    walking the million iterations (it was 1.7 s of a warp and the tail of the whole bench pass: DESIGN.md 4.1/5).
    Column 84815 of shard 4 of the C4 bench ensemble, found with tests/gpu_diag_tile.py."""
    from lgar_b200 import workloads, forward_raw, STATUS_NAMES
    from oracle import lgar_oracle as O
    T, b = 8760, 84815
    we = workloads.synthetic_sites_ensemble(B=125_000, T=T, sites=128, rank=4, shared_sites=True)
    cols = np.array([b] * 32)
    ens = _ens(we, cols)
    a, n, k = (np.ascontiguousarray(x[:, cols]) for x in (we.alpha, we.n, we.ksat))
    res, ws = forward_raw(ens, a, n, k, outputs=(), per_step=False, window=(0, 8640), counters=True)
    torch.cuda.synchronize()
    before = res.counters.cpu().numpy().astype(np.int64)
    assert (res.status.cpu().numpy() == 0).all()
    res, ws = forward_raw(ens, a, n, k, outputs=(), per_step=False, workspace=ws, window=(8640, T), into=res, counters=True)
    torch.cuda.synchronize()
    st, cr = res.status.cpu().numpy(), res.crash_step.cpu().numpy()
    cfg = O.make_cfg(we.alpha[:, b], we.n[:, b], we.ksat[:, b], we.theta_r[:, b], we.theta_e[:, b], thickness=we.thickness[:, b],
                     iter_cap=1_000_000)
    r = O.forward(cfg, we.forcing[we.site_index[b]], fronts=False)
    assert STATUS_NAMES[int(r["status"])] == "ITER_CAP"
    assert (st == r["status"]).all() and (cr == r["crash_step"]).all(), (st[:2], cr[:2], r["status"], r["crash_step"])
    colmass = int(res.counters.cpu().numpy()[6])  # check_column_mass evaluations of the last 120 rows, 32 lanes
    assert colmass < 32 * 20_000, f"{colmass} column-mass evaluations: the flat run was walked, not jumped"
    del before
