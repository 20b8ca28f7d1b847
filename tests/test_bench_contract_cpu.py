"""The reference arm of bench.py (`--impl reference`) runs on host cores only, so its JSON contract can be checked
without a GPU: one line, the keys the driver reads, `impl: reference`, a cpu_baseline block describing the run and an
e2e block that repeats the value with zero transfer bytes.  With the Python reference present (/root/reference in the
build container, oracle/_ref on the GPU box) the line's value is the unmodified reference (kind "reference") and the
C++ restatement is reported beside it (`port`); without it (--no-pyref) the port is the value (kind "port")."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--gpus", "1", "--steps", "1", "--warmup", "1", "--columns", "256", "--nsteps", "240", "--sites", "4",
         "--cpu-sample-columns", "32"]


def _run(extra, env=None, timeout=900):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *extra],
                         capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    return [l for l in out.stdout.splitlines() if l.startswith("{")]


def _common(d):
    assert d["impl"] == "reference" and d["metric"].startswith("column-timesteps/sec")
    assert d["unit"] == "column-timesteps/s" and d["higher_is_better"] is True and d["n_gpus"] == 1
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and "workload" in d["config"]
    assert d["cpu_baseline"]["value"] == d["value"] and d["cpu_baseline"]["cores"] >= 1


def test_reference_arm_port_only():
    lines = _run(SMALL + ["--no-pyref"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    _common(d)
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and "32 columns" in cb["sample"] and "alive column-steps" in cb["sample"]
    assert d["fwd_grad"]["value"] > 0


def test_reference_arm_python_reference():
    have = any(os.path.isdir(os.path.join(p, "dpLGAR")) for p in ("/root/reference", os.path.join(ROOT, "oracle", "_ref")))
    lines = _run(SMALL + ["--pyref-rows", "24", "--pyref-procs", "2"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    _common(d)
    if have:
        assert d["cpu_baseline"]["kind"] == "reference" and "unmodified Python reference" in d["cpu_baseline"]["sample"]
        assert d["port"]["kind"] == "port" and d["port"]["value"] > d["value"]
        assert d["fwd_grad"]["value"] > 0
    else:
        assert d["cpu_baseline"]["kind"] == "port"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_segments_cover_the_record_once():
    sys.path.insert(0, ROOT)
    import bench
    for T, K in ((8760, 20), (8760, 7), (8760, 1000), (8760, 8760), (100, 20), (5, 20), (64, 1)):
        segs = bench.segments(T, K)
        assert segs[0][0] == 0 and segs[-1][1] == T and len(segs) == min(K, T)
        assert all(a[1] == b[0] for a, b in zip(segs, segs[1:])) and all(t1 > t0 for t0, t1 in segs)
        assert max(t1 - t0 for t0, t1 in segs) == segs[0][1] - segs[0][0]  # the e2e staging buffers are sized by it


def test_steps_beyond_the_record_are_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--nsteps", "10", "--steps", "11"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


def _result(B, T, seed, crashed_fraction):
    """A ForwardResult shaped like the library's: a crashed column has NaN in every row from its crash step on and,
    like a column ending in status NAN, NaN sums."""
    import torch
    from lgar_b200 import ForwardResult, output_mask
    g = torch.Generator().manual_seed(seed)
    f64 = dict(generator=g, dtype=torch.float64)
    crashed = torch.rand(B, **f64) < crashed_fraction
    status = torch.where(crashed, torch.randint(1, 9, (B,), generator=g, dtype=torch.int32), 0).to(torch.int32)
    crash_step = torch.where(crashed, torch.randint(0, T, (B,), generator=g, dtype=torch.int32), -1).to(torch.int32)
    per_step = torch.rand((2, T, B), **f64)
    per_step[:, torch.arange(T)[:, None] >= torch.where(crashed, crash_step, T)[None, :]] = float("nan")
    sums = torch.rand((10, B), **f64)
    sums[:, crashed] = float("nan")
    return ForwardResult(per_step=per_step, mask=output_mask(("runoff", "AET")), sums=sums,
                         start_volume=torch.rand(B, **f64), status=status, crash_step=crash_step)


def _load(d, name):
    """A dumped float array with its no-value entries restored to NaN."""
    v, m = np.load(d / f"{name}.npy"), np.load(d / f"{name}_nonfinite.npy")
    assert v.dtype == np.float64 and m.dtype == np.float32 and v.shape == m.shape and np.isin(m, (0, 1)).all()
    assert (v[m == 1] == 0).all()
    return np.where(m == 1, np.nan, v)


def _idx(d, name):
    i = np.load(d / f"{name}.npy")
    assert i.dtype == np.float64 and (np.diff(i) > 0).all()
    return i.astype(np.int64)


def test_dump_outputs_sample_and_budget(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    B, T, outs, budget = 3000, 40, ("runoff", "AET"), 400_000
    res = _result(B, T, seed=0, crashed_fraction=0.3)
    monkeypatch.setattr(bench, "DUMP_BYTES", budget)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, (25, 40), outs)
    a = tmp_path / "a"
    files = sorted(p.name[:-4] for p in a.iterdir())
    assert files == sorted(["AET", "AET_nonfinite", "columns", "crash_step", "runoff", "runoff_nonfinite", "series_columns",
                            "series_rows", "start_volume", "start_volume_nonfinite", "status", "sums", "sums_nonfinite"])
    total = 0
    for f in files:
        x, y = np.load(a / f"{f}.npy"), np.load(tmp_path / "b" / f"{f}.npy")
        assert x.dtype in (np.float32, np.float64) and np.isfinite(x).all(), f
        assert np.array_equal(x, y)  # the same sample every time
        total += x.nbytes
    assert total <= budget
    cols, rows, scols = _idx(a, "columns"), _idx(a, "series_rows"), _idx(a, "series_columns")
    assert 0 < len(cols) < B and 0 < len(scols) < B and cols[-1] < B and scols[-1] < B
    assert rows.tolist() == list(range(25, 40))
    # the values as the library returned them, NaN of the crashed columns included
    np.testing.assert_array_equal(np.load(a / "status.npy"), res.status[cols].numpy())
    np.testing.assert_array_equal(np.load(a / "crash_step.npy"), res.crash_step[cols].numpy())
    np.testing.assert_array_equal(_load(a, "start_volume"), res.start_volume[cols].numpy())
    np.testing.assert_array_equal(_load(a, "sums"), res.sums[:, cols].numpy())
    assert np.isnan(_load(a, "sums")).any() and np.isnan(_load(a, "runoff")).any()
    for q, name in enumerate(outs):
        np.testing.assert_array_equal(_load(a, name), res.per_step[q][rows][:, scols].numpy())


def test_dump_sample_does_not_depend_on_the_results(tmp_path, monkeypatch):
    """Two results that differ in one column (it ends in ITER_CAP instead of OK) give the same sampled elements:
    everything but that column's entries compares equal, so a one-column change shows as one column."""
    sys.path.insert(0, ROOT)
    import bench
    B, T, outs = 3000, 40, ("runoff", "AET")
    monkeypatch.setattr(bench, "DUMP_BYTES", 400_000)
    r1 = _result(B, T, seed=2, crashed_fraction=0.3)
    bench.dump_outputs(str(tmp_path / "a"), r1, (25, 40), outs)
    cols, scols = _idx(tmp_path / "a", "columns"), _idx(tmp_path / "a", "series_columns")
    ok = r1.status.numpy() == 0
    b = int(np.intersect1d(cols[ok[cols]], scols)[0])  # an OK column in both samples
    r2 = _result(B, T, seed=2, crashed_fraction=0.3)
    r2.status[b], r2.crash_step[b] = 7, 30
    r2.per_step[:, 30:, b] = float("nan")
    r2.sums[:, b] = float("nan")
    bench.dump_outputs(str(tmp_path / "b"), r2, (25, 40), outs)
    for f in ("columns", "series_rows", "series_columns"):
        np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{f}.npy"), np.load(tmp_path / "b" / f"{f}.npy"))
    for name, ix in (("status", cols), ("sums", cols), ("runoff", scols), ("AET", scols)):
        x = np.load(tmp_path / "a" / "status.npy") if name == "status" else _load(tmp_path / "a", name)
        y = np.load(tmp_path / "b" / "status.npy") if name == "status" else _load(tmp_path / "b", name)
        assert x.shape == y.shape
        same = ((x == y) | (np.isnan(x) & np.isnan(y))).reshape(-1, x.shape[-1]).all(axis=0)  # per sampled column
        assert ix[~same].tolist() == [b], name


def test_dump_outputs_keeps_everything_that_fits(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    B, T = 50, 12
    res = _result(B, T, seed=1, crashed_fraction=0.2)
    assert 0 < (res.status.numpy() == 0).sum() < B
    bench.dump_outputs(str(tmp_path), res, (8, 12), ("runoff", "AET"))
    assert _idx(tmp_path, "columns").tolist() == list(range(B)) == _idx(tmp_path, "series_columns").tolist()
    assert _idx(tmp_path, "series_rows").tolist() == [8, 9, 10, 11]
    np.testing.assert_array_equal(np.load(tmp_path / "status.npy"), res.status.numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "crash_step.npy"), res.crash_step.numpy())
    np.testing.assert_array_equal(_load(tmp_path, "sums"), res.sums.numpy())
    np.testing.assert_array_equal(_load(tmp_path, "runoff"), res.per_step[0, 8:12].numpy())
    np.testing.assert_array_equal(_load(tmp_path, "AET"), res.per_step[1, 8:12].numpy())


def test_dump_outputs_is_rejected_with_the_reference_arm():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
