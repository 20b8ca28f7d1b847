"""-m gpu: the launches bench.py times.

* A record advanced window by window (lgar_problem.step_begin / step_end, the bench's "steps") gives the bits of ONE
  launch over the whole record: per-step series, sums, status, crash step -- for windows that do not align with the
  scheduler's chunks, and for the window sizes the bench uses.
* bench.py --dump-outputs writes the bits of the timed pass's last window.
* lgar_forward_host (the host-pointer entry of the C ABI) gives the bits of the device-pointer entry.
* The C ABI rejects windows that cannot work (no resume, keep_checkpoints, out of range)."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
OUTS = ("runoff", "AET", "ending_volume")


def _setup(B=4097, T=300, sites=4, rank=1, **kw):
    from lgar_b200 import workloads, ColumnEnsemble
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=sites, rank=rank)
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, **kw)
    return we, ens


@pytest.mark.parametrize("nseg", [2, 7, 20])
def test_windows_equal_one_launch(nseg):
    from lgar_b200 import forward_raw
    import bench
    we, ens = _setup()
    T = ens.num_steps
    full, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUTS, num_fronts=True)
    res, ws = None, None
    for (t0, t1) in bench.segments(T, nseg):
        res, ws = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUTS, num_fronts=True, workspace=ws, window=(t0, t1), into=res)
    torch.cuda.synchronize()
    assert torch.equal(res.status, full.status)
    assert (full.status != 0).any(), "the case must contain crashing columns"
    c_full = full.crash_step.cpu().numpy()
    c_win = res.crash_step.cpu().numpy()
    c_win = np.where(c_win <= -2, -2 - c_win, c_win)  # crashed in an earlier window: -2 - t
    np.testing.assert_array_equal(c_win, c_full)
    ok = full.status == 0
    assert torch.equal(res.sums[:, ok].contiguous().view(torch.int64), full.sums[:, ok].contiguous().view(torch.int64))
    # crashed columns: sums of the completed steps are identical too
    assert torch.equal(res.sums[:4, ~ok].contiguous().view(torch.int64), full.sums[:4, ~ok].contiguous().view(torch.int64))
    a, b = res.per_step.view(torch.int64), full.per_step.view(torch.int64)  # NaN rows after a crash compare by bits
    assert torch.equal(a, b)
    assert torch.equal(res.num_fronts, full.num_fronts)
    assert np.array_equal(bench.alive_steps_of(res.status.cpu().numpy(), res.crash_step.cpu().numpy(), T),
                          bench.alive_steps_of(full.status.cpu().numpy(), c_full, T))


@pytest.mark.parametrize("B,chunk", [(40_000, 16), (40_000, 64), (4097, 64)])
def test_pipelined_windows_equal_one_launch(B, chunk):
    """Consecutive windows launched as a pipelined sequence (programmatic dependent launch, lgar_problem.pipeline_seq):
    window k+1 runs while window k drains; the per-tile progress counters order the column states.  40,000 columns fill
    the device (the overlapped path); 4097 columns do not (the library falls back to stream-ordered launches)."""
    from lgar_b200 import forward_raw
    import bench
    we, ens = _setup(B=B, T=200, sites=8, rank=2, chunk_steps=chunk)
    T = ens.num_steps
    full, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUTS)
    for rep in range(2):   # the second sequence reuses the workspace (ticket epochs restart at 1)
        res, ws = None, None
        for i, (t0, t1) in enumerate(bench.segments(T, 5)):
            res, ws = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUTS, workspace=ws, window=(t0, t1), into=res,
                                  pipeline_seq=i + 1)
        torch.cuda.synchronize()
        assert torch.equal(res.status, full.status)
        assert torch.equal(res.sums.view(torch.int64), full.sums.view(torch.int64))
        assert torch.equal(res.per_step.view(torch.int64), full.per_step.view(torch.int64))
        c = res.crash_step.cpu().numpy()
        np.testing.assert_array_equal(np.where(c <= -2, -2 - c, c), full.crash_step.cpu().numpy())


def test_bench_steps_and_dumped_outputs(tmp_path):
    """bench.py --steps K times K launches, and --dump-outputs writes what the last one returned: the rows of its window
    and the per-column results, equal to one launch over the whole record of the same shard and placement."""
    import json
    import os
    import subprocess
    import sys
    from lgar_b200 import forward_raw, workloads, ColumnEnsemble
    import bench
    B, T, K, sites = 4096, 240, 7, 4
    root = os.path.dirname(os.path.abspath(bench.__file__))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", str(K), "--warmup", "2",
                          "--columns", str(B), "--nsteps", str(T), "--sites", str(sites), "--no-cpu-baseline", "--no-e2e",
                          "--grad-columns", "0", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == K and line["gpu_launches"] == K
    we = workloads.synthetic_sites_ensemble(B=B, T=T, sites=sites, rank=0, shared_sites=True)
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, max_fronts=16, chunk_steps=64, device="cuda:0")
    ksat = torch.from_numpy(we.ksat).cuda()
    ens.balance(ksat)
    full, _ = forward_raw(ens, we.alpha, we.n, ksat, outputs=("runoff", "AET"))
    torch.cuda.synchronize()
    t0 = bench.segments(T, K)[-1][0]
    bits = lambda a: np.ascontiguousarray(a).view(np.int64)
    load = lambda f: np.load(tmp_path / f"{f}.npy")
    assert all(np.isfinite(np.load(f)).all() for f in tmp_path.iterdir())
    status = full.status.cpu().numpy()
    assert 0 < (status == 0).sum() < B, "the case must contain crashing columns"
    # all 4096 columns and every row of the last window fit
    np.testing.assert_array_equal(load("columns"), np.arange(B))
    np.testing.assert_array_equal(load("series_columns"), np.arange(B))
    np.testing.assert_array_equal(load("series_rows"), np.arange(t0, T))
    np.testing.assert_array_equal(load("status"), status)
    c = load("crash_step")
    np.testing.assert_array_equal(np.where(c <= -2, -2 - c, c), full.crash_step.cpu().numpy())
    for name, want in (("start_volume", full.start_volume), ("sums", full.sums),
                       ("runoff", full["runoff"][t0:]), ("AET", full["AET"][t0:])):
        want = want.cpu().numpy()
        missing = load(f"{name}_nonfinite") == 1
        np.testing.assert_array_equal(missing, ~np.isfinite(want))  # the NaN after a crash step, exactly there
        np.testing.assert_array_equal(bits(load(name)[~missing]), bits(want[~missing]))


def test_window_argument_checks():
    from lgar_b200 import forward_raw, LGARLibraryError
    we, ens = _setup(B=64, T=50, sites=1)
    with pytest.raises(LGARLibraryError):   # does not start at row 0 without a previous state ... resume is implied, but
        forward_raw(ens, we.alpha, we.n, we.ksat, window=(10, 60))          # ... the window leaves the record
    with pytest.raises(LGARLibraryError):
        forward_raw(ens, we.alpha, we.n, we.ksat, window=(20, 20))
    with pytest.raises(LGARLibraryError):
        forward_raw(ens, we.alpha, we.n, we.ksat, window=(0, 25), keep_checkpoints=True)


def test_forward_host_entry_point():
    """lgar_forward_host: every pointer is a HOST pointer; the library stages, runs and copies back."""
    from lgar_b200 import forward_raw, _capi, output_mask, OUT_NAMES
    we, ens = _setup(B=333, T=90, sites=2, rank=5)
    ref, _ = forward_raw(ens, we.alpha, we.n, we.ksat, outputs=OUT_NAMES, num_fronts=True)
    torch.cuda.synchronize()
    B, T, L = 333, 90, 3
    keep = []

    def hp(a, dt=np.float64):
        a = np.ascontiguousarray(a, dtype=dt)
        keep.append(a)
        return a.ctypes.data
    p = ens.problem(torch.zeros(1), torch.zeros(1), torch.zeros(1))
    p.alpha, p.n, p.ksat = hp(we.alpha), hp(we.n), hp(we.ksat)
    p.theta_r, p.theta_e, p.thickness = hp(we.theta_r), hp(we.theta_e), hp(we.thickness)
    p.initial_psi, p.ponded_depth_max = hp(np.full(B, 2000.0)), hp(np.zeros(B))
    p.forcing, p.site_index = hp(we.forcing), hp(we.site_index, np.int32)
    o = _capi.Outputs()
    mask = output_mask(OUT_NAMES)
    per_step = np.empty((len(OUT_NAMES), T, B)); sums = np.empty((len(OUT_NAMES), B)); sv = np.empty(B)
    st = np.empty(B, dtype=np.int32); cs = np.empty(B, dtype=np.int32); nf = np.empty((T, B), dtype=np.int32)
    o.per_step, o.per_step_mask, o.sums, o.start_volume = per_step.ctypes.data, mask, sums.ctypes.data, sv.ctypes.data
    o.status, o.crash_step, o.num_fronts = st.ctypes.data, cs.ctypes.data, nf.ctypes.data
    _capi.check(_capi.lib().lgar_forward_host(C.byref(p), C.byref(o)), "lgar_forward_host")
    np.testing.assert_array_equal(st, ref.status.cpu().numpy())
    np.testing.assert_array_equal(cs, ref.crash_step.cpu().numpy())
    np.testing.assert_array_equal(nf, ref.num_fronts.cpu().numpy())
    np.testing.assert_array_equal(sums.view(np.int64), ref.sums.cpu().numpy().view(np.int64))
    np.testing.assert_array_equal(per_step.view(np.int64), ref.per_step.cpu().numpy().view(np.int64))
    np.testing.assert_array_equal(sv, ref.start_volume.cpu().numpy())
