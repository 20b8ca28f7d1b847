#!/usr/bin/env python
"""bench.py -- column-timesteps/sec of the LGAR time-stepping core on N B200s.

Workload (config C4 of BASELINE.json, one GPU's share): 125,000 columns x 8760 hourly steps, 3 layers,
128 synthetic site records per GPU, per-column random van Genuchten parameters.  `--workload c3` selects
config C3 instead (Bushland record, 100,000-member parameter ensemble, forward only).  Weak scaling: every
rank draws its own shard; no data-path collective (columns are independent).

A bench "step" is ONE TIME SEGMENT of the record: the whole shard advanced through ceil(T / steps) or
floor(T / steps) consecutive forcing rows (steps <= T) by one persistent launch (`lgar_problem.step_begin/step_end`,
continuing from the column state the previous launch left in the workspace -- the way the reference's training loop feeds
dpLGAR.forward one row after the other, agents/DifferentiableLGAR.py:117-125).  The K timed steps together
are exactly ONE pass over the full record (results bit-identical to a single launch: tests/test_gpu_bench_path.py);
the W warm-up steps run the first W segments and the timed pass then restarts from the initial state.

  python bench.py --gpus 1 --steps K --warmup W            # CUDA path (this repo)
  python bench.py --impl reference ...                     # the reference on the box's host cores
  python bench.py ... --dump-outputs DIR                   # + what the last timed step returned, as DIR/*.npy

`value`   : whole-job column-timesteps/s, inputs resident in HBM, CUDA-event time, max over ranks.  Only
            column-steps that were actually simulated count: a column the reference would abort with an
            exception stops at its crash step (config.status_histogram) -- same definition in every arm.
`e2e`     : the same pass through the public API (lgar_b200.forward_raw) with HOST (pinned) parameters and
            forcing: every step copies its forcing segment H2D (step 0: the parameters too) and copies the
            per-step series it produced (runoff, AET) plus, at the end, sums/status/crash_step D2H.
`fwd_grad`: forward (with checkpoints) + hand-written reverse kernel over the WHOLE shard and record,
            loss = mean over OK columns of sum_t (runoff_t + AET_t)   (agents/DifferentiableLGAR.py:163).
`roofline`: FP64-ALU bound (SURVEY 8d): algorithmic flop counted from closure-call counters.
`parity`  : the first columns of the shard against the CPU oracle (the cpu_baseline leg computes them anyway).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "column-timesteps/sec (fwd)"
UNIT = "column-timesteps/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c3"])
    ap.add_argument("--columns", type=int, default=0, help="columns per GPU (default: 125000 for c4, 100000 for c3)")
    ap.add_argument("--nsteps", type=int, default=8760, help="forcing steps T of the record")
    ap.add_argument("--sites", type=int, default=128, help="forcing records per GPU (c4)")
    ap.add_argument("--max-fronts", type=int, default=16)
    ap.add_argument("--chunk", type=int, default=64)
    ap.add_argument("--cpu-sample-columns", type=int, default=0)
    ap.add_argument("--count-fraction", type=float, default=0.25,
                    help="fraction of the 32-column tiles run through the counting kernel (algorithmic flop)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="A/B: stream-ordered windows (no programmatic dependent launch)")
    ap.add_argument("--e2e-interleaved", action="store_true", help="A/B: D2H of every segment right behind its launch")
    ap.add_argument("--no-balance", action="store_true", help="A/B: identity placement of columns on warps")
    ap.add_argument("--no-pyref", action="store_true", help="reference arm: skip the Python reference (port only)")
    ap.add_argument("--pyref-rows", type=int, default=0, help="reference arm: forcing rows per step of the Python reference")
    ap.add_argument("--pyref-procs", type=int, default=0, help="reference arm: processes of the Python reference (default min(8, cores))")
    ap.add_argument("--shard-rank", type=int, default=-1,
                    help="diagnosis: run the shard of this rank of a multi-GPU job on a single GPU (shard vs GPU differences)")
    ap.add_argument("--rank-sites", action="store_true",
                    help="A/B: every rank draws its own site records too (shards then differ in work by several per cent)")
    ap.add_argument("--grad-columns", type=int, default=-1,
                    help="columns of the shard used for the forward+gradient figure (-1 = the whole shard, 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned as DIR/<name>.npy (at most 64 MB in all, a sample "
                         "with a fixed seed where the shard does not fit, sampled indices beside it); rank 0's shard")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the results of the CUDA path (--impl b200)")
    if args.impl == "b200" and args.steps > args.nsteps:
        ap.error("--steps must not exceed --nsteps: every timed step advances the shard by at least one forcing row")
    if args.columns <= 0:
        args.columns = 125_000 if args.workload == "c4" else 100_000
    if args.workload == "c3":
        args.sites = 1
        if args.grad_columns < 0:
            args.grad_columns = 0  # C3 is forward only (BASELINE.json configs[2])
    if args.grad_columns < 0:
        args.grad_columns = args.columns
    return args


def workload_name(args):
    if args.workload == "c3":
        return (f"C3: Bushland resampled forcing, {args.columns}-member parameter ensemble per GPU x {args.nsteps} hourly "
                "steps, 3 layers, forward only, alpha~U[0.0015,0.015] n~U[1.1,3] Ks~logU[0.01,30]")
    return (f"C4 shard per GPU: {args.columns} columns x {args.nsteps} hourly steps, 3 layers, {args.sites} synthetic "
            "sites, alpha~U[0.0015,0.015] n~U[1.1,3] Ks~logU[0.01,30]"
            + ("; N-GPU job: every rank draws its own site records too" if args.rank_sites else
               "; N-GPU job: the same site records on every rank, own parameter members (equivalent shards)")
            + (f" (shard of rank {args.shard_rank})" if args.shard_rank >= 0 else ""))


def make_workload(args, rank):
    from lgar_b200 import workloads
    if args.workload == "c3":
        return workloads.bushland_ensemble(B=args.columns, T=args.nsteps, seed=rank)
    return workloads.synthetic_sites_ensemble(B=args.columns, T=args.nsteps, sites=args.sites, rank=rank,
                                              shared_sites=not args.rank_sites)


def segments(T, steps):
    """min(steps, T) consecutive non-empty windows [t0, t1) that cover the record once; the first is the longest."""
    k = min(steps, T)
    b = [-(-i * T // k) for i in range(k + 1)]
    return list(zip(b[:-1], b[1:]))


DUMP_BYTES = 63 * 10**6  # array data; the .npy headers fit in what is left of 64 MB


def _sample(n, k, seed):
    """Sorted indices of k of range(n), drawn with a fixed seed; all of range(n) when k >= n."""
    if k >= n:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, max(k, 1), replace=False))


def dump_outputs(path, res, window, outs):
    """--dump-outputs: what the last timed step returned to its caller, as .npy files of at most DUMP_BYTES in all.
    Per column (indices in `columns`): `status`, `crash_step`, `start_volume` and `sums` [10, C] (running totals of all
    outputs since row 0).  Per step: the series `outs` over the step's window, one [rows, C'] file each (absolute rows
    in `series_rows`, columns in `series_columns`).  Where a whole array does not fit, a sample drawn from the shape
    alone with a fixed seed stands for it, so that two builds run with the same arguments write the same elements
    whatever their results.  A column the reference aborts has no values from its crash step on, which the library
    marks NaN: every float array is written as float64 with such entries set to 0, beside a float32 `<name>_nonfinite`
    that is 1 exactly there, so the files hold finite numbers and lose nothing."""
    import torch
    os.makedirs(path, exist_ok=True)
    dev = res.status.device
    B, nout = res.status.numel(), res.sums.shape[0]

    def save(name, v, dtype=torch.float64):
        np.save(os.path.join(path, f"{name}.npy"), v.to(dtype).cpu().numpy())

    def save_values(name, v):
        finite = torch.isfinite(v)
        save(name, torch.where(finite, v, torch.zeros_like(v)))
        save(f"{name}_nonfinite", ~finite, torch.float32)

    def sample(n, k, seed):
        return torch.from_numpy(_sample(n, k, seed)).to(dev)

    per_column = 8 * (3 + nout + 1) + 4 * (1 + nout)  # status, crash step, start volume, sums, index; two masks
    cols = sample(B, DUMP_BYTES // 2 // per_column, seed=1)
    save("columns", cols)
    save("status", res.status.index_select(0, cols))
    save("crash_step", res.crash_step.index_select(0, cols))
    save_values("start_volume", res.start_volume.index_select(0, cols))
    save_values("sums", res.sums.index_select(1, cols))
    left = DUMP_BYTES - per_column * cols.numel()
    t0, t1 = window
    per_element = 12 * len(outs)  # float64 value + float32 mask of every series
    rows = t0 + sample(t1 - t0, (left - 8) // (per_element + 8), seed=2)  # leaves room for at least one column
    series_cols = sample(B, (left - 8 * rows.numel()) // (per_element * rows.numel() + 8), seed=3)
    save("series_rows", rows)
    save("series_columns", series_cols)
    for name in outs:
        save_values(name, res[name].index_select(0, rows).index_select(1, series_cols))


def alive_steps_of(status, crash, T):
    """Column-steps actually simulated: T for an OK column, the number of completed steps for a column the
    reference aborts (crash_step; -2 - t encodes 'crashed at step t of an earlier window')."""
    crash = np.where(crash <= -2, -2 - crash, crash)
    return np.where(status == 0, T, np.clip(crash, 0, T))


class ClockSampler(threading.Thread):
    """SM clock / power / throttle reasons of one GPU during the timed region, through NVML in-process
    (no nvidia-smi fork per sample); falls back to nvidia-smi at a low rate if NVML is unavailable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake"}

    def __init__(self, cuda_index=0, interval=0.25):
        super().__init__(daemon=True)
        self.interval = interval
        self.rows = []          # (sm_mhz, power_w, reasons_bitmask)
        self.stop_flag = False
        self.max_mhz = None
        self.index = cuda_index
        self.handle = None
        self.nv = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(cuda_index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.handle, self.nv = h, nv
        except Exception:
            self.handle = None

    def _sample_nvml(self):
        nv, h = self.nv, self.handle
        mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
        try:
            pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
        except Exception:
            pw = float("nan")
        try:
            rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
        except Exception:
            try:
                rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            except Exception:
                rs = 0
        self.rows.append((mhz, pw, rs))

    def _sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        if len(r) >= 7:
            bits = sum(b for b, on in zip((0x8, 0x40, 0x20, 0x4), r[3:7]) if on == "Active")
            self.max_mhz = float(r[1])
            self.rows.append((float(r[0]), float(r[2]) if r[2].replace(".", "").isdigit() else float("nan"), bits))

    def run(self):
        while not self.stop_flag:
            try:
                if self.handle is not None:
                    self._sample_nvml()
                else:
                    self._sample_smi()
            except Exception:
                pass
            time.sleep(self.interval if self.handle is not None else max(self.interval, 2.0))

    def summary(self):
        sm = [r[0] for r in self.rows]
        pw = [r[1] for r in self.rows if r[1] == r[1]]
        bits = 0
        for r in self.rows:
            bits |= r[2]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz,
                "sm_mhz_min": float(min(sm)) if sm else None, "power_w": float(np.median(pw)) if pw else None,
                "reasons": [nm for b, nm in self.REASONS.items() if bits & b], "samples": len(self.rows),
                "source": "nvml" if self.handle is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------------
# CPU arms (oracle/ is test infrastructure: only these legs and the tests may execute it)
# ---------------------------------------------------------------------------------------------------------
def oracle_cfgs(we, idx):
    from oracle import lgar_oracle as O
    # iter_cap: the CUDA path's default (lgar_problem.iter_cap = 0 -> 1,000,000), so that both arms cut the same columns
    return [O.make_cfg(we.alpha[:, b], we.n[:, b], we.ksat[:, b], we.theta_r[:, b], we.theta_e[:, b],
                       thickness=we.thickness[:, b], iter_cap=1_000_000) for b in idx]


def port_run(we, idx, T, threads, tangents=False):
    """The C++ restatement of the reference (oracle/, kind='port') on columns `idx`, all host threads.
    Returns (alive column-steps simulated, seconds, result dict)."""
    from oracle import lgar_oracle as O
    cfgs = oracle_cfgs(we, idx)
    t0 = time.perf_counter()
    r = O.forward_batch_ex(cfgs, we.forcing[:, :T], we.site_index[idx], nthreads=threads, tangents=tangents)
    dt = time.perf_counter() - t0
    alive = int(alive_steps_of(r["status"], r["crash_step"], T).sum())
    return alive, dt, r


def pyref_run(we, args, nproc, rows_timed, rows_warm, grad, budget_s=60.0):
    """The UNMODIFIED Python reference (oracle/_ref or /root/reference) on columns 0..nproc-1 of the ensemble,
    one process x one thread per column.  Returns dict or None if the reference is not available."""
    ref_ok = any(os.path.isdir(os.path.join(p, "dpLGAR")) for p in ("/root/reference", os.path.join(ROOT, "oracle", "_ref")))
    if not ref_ok:
        return None
    tmp = tempfile.mkdtemp(prefix="lgar_pyref_")
    procs = []
    rows = min(rows_warm + rows_timed, args.nsteps)
    kinds = ("phil", "bush")
    for i in range(nproc):
        b = i * (we.num_columns // nproc)  # spread over the shard (different sites)
        site = int(we.site_index[b])
        kind = "bush" if args.workload == "c3" else kinds[site % 2]
        spec = os.path.join(tmp, f"col{i}.npz")
        np.savez(spec, forcing=we.forcing[site, :rows], alpha=we.alpha[:, b], n=we.n[:, b], ksat=we.ksat[:, b],
                 soil_rows=np.array([12, 13, 14] if kind == "phil" else [15, 16, 17]))
        cmd = [sys.executable, os.path.join(ROOT, "oracle", "time_reference.py"), "--spec", spec, "--warm-rows", str(rows_warm),
               "--budget-s", str(budget_s)] + (["--grad"] if grad else [])
        env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", CUDA_VISIBLE_DEVICES="")
        procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env))
    res = []
    for p in procs:
        try:
            out, err = p.communicate(timeout=budget_s + 240)
            lines = [l for l in out.splitlines() if l.startswith("{")]
            if p.returncode == 0 and lines:
                res.append(json.loads(lines[-1]))
        except Exception:
            p.kill()
    if not res:
        return None
    steps = sum(r["steps"] for r in res)
    secs = max(r["seconds"] for r in res)
    return {"value": steps / secs if secs > 0 else 0.0, "processes": len(res), "column_steps": steps, "seconds": secs,
            "per_core": float(np.mean([r["steps"] / r["seconds"] for r in res if r["seconds"] > 0])),
            "crashed_columns": sum(1 for r in res if r["crash"]), "ref_root": res[0]["ref_root"]}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores.

    value / cpu_baseline (kind 'reference'): the UNMODIFIED Python reference staged in oracle/_ref (oracle/make_ref.sh),
    min(8, cores) processes x 1 thread, one column of the ensemble each; a bench step = `rows_per_step` forcing rows on
    every process (W warm-up steps, then K timed steps).  `port`: the validated C++ restatement (oracle/lgar_oracle.cpp,
    pinned bit-for-bit to the Python reference's goldens) on all host threads -- a second, much stronger CPU figure;
    it becomes `value` only if the Python reference is not present."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    we = make_workload(args, 0)
    threads = os.cpu_count() or 1
    T = args.nsteps
    line = {
        "impl": "reference", "metric": METRIC, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(args)},
    }
    # ---- the Python reference ------------------------------------------------------------------------
    py = pyg = None
    if not args.no_pyref:
        nproc = args.pyref_procs or max(1, min(8, threads))
        rows_per_step = args.pyref_rows or max(12, int(round(240 / args.steps)))
        rows_timed, rows_warm = rows_per_step * args.steps, rows_per_step * args.warmup
        both = threads >= 2 * nproc
        if both:  # forward and forward+gradient sets side by side (one core each)
            box = {}
            th = threading.Thread(target=lambda: box.update(g=pyref_run(we, args, nproc, rows_timed, rows_warm, True)))
            th.start()
            py = pyref_run(we, args, nproc, rows_timed, rows_warm, False)
            th.join()
            pyg = box.get("g")
        else:
            py = pyref_run(we, args, nproc, rows_timed, rows_warm, False)
            pyg = pyref_run(we, args, nproc, rows_timed, rows_warm, True)
    # ---- the C++ port ----------------------------------------------------------------------------------
    ncol = min(args.cpu_sample_columns or 8 * threads, we.num_columns)
    B = we.num_columns
    for w in range(min(args.warmup, 2)):
        port_run(we, np.arange(min(ncol, 2 * threads)), min(T, 200), threads)
    alive_tot, secs = 0, []
    for i in range(args.steps):  # a different block of columns every step: the sample covers steps * ncol columns
        idx = (np.arange(ncol) + i * ncol) % B
        alive, dt, _ = port_run(we, idx, T, threads)
        alive_tot += alive
        secs.append(dt)
    port_val = alive_tot / sum(secs)
    gcol = max(threads, ncol // 4)
    g_alive, g_dt, _ = port_run(we, np.arange(gcol), T, threads, tangents=True)
    port = {"value": port_val, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{ncol} columns x {T} steps per step, {args.steps} disjoint column blocks of the same ensemble, "
                      f"alive column-steps only ({sum(secs):.1f} s)",
            "fwd_grad": {"value": g_alive / g_dt, "what": f"forward-mode tangents w.r.t. 9 parameters, {gcol} columns x {T} steps"}}
    if py:
        value = py["value"]
        sample = (f"{py['processes']} columns (one per process, 1 thread each) x {rows_per_step} forcing rows per step, "
                  f"{args.warmup} warm-up + {args.steps} timed steps from the initial state; unmodified Python reference "
                  f"({os.path.relpath(py['ref_root'], ROOT) if py['ref_root'].startswith(ROOT) else py['ref_root']}), "
                  f"torch.no_grad, {py['per_core']:.1f} column-steps/s per core")
        line.update(value=value, ms_per_step=py["seconds"] / args.steps * 1e3)
        line["cpu_baseline"] = {"value": value, "unit": UNIT, "cores": py["processes"], "kind": "reference", "sample": sample}
        if pyg:
            line["fwd_grad"] = {"value": pyg["value"], "unit": UNIT, "per_core": pyg["per_core"],
                                "what": "autograd graph + loss.backward(), loss = sum_t (runoff + AET), same columns and rows"}
        line["port"] = port
    else:
        line.update(value=port_val, ms_per_step=float(np.mean(secs)) * 1e3)
        line["cpu_baseline"] = port
        line["fwd_grad"] = {"value": port["fwd_grad"]["value"], "unit": UNIT, "what": port["fwd_grad"]["what"]}
    line["config"]["sample"] = line["cpu_baseline"]["sample"]
    line["e2e"] = {"value": line["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
        return
    t_start = time.perf_counter()
    import torch
    import torch.distributed as dist
    import lgar_b200  # noqa: F401
    from lgar_b200 import workloads, ColumnEnsemble, forward_raw, _capi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _capi.check(_capi.lib().lgar_device_check(), "lgar_device_check")

    B, T = args.columns, args.nsteps
    we = make_workload(args, rank if args.shard_rank < 0 else args.shard_rank)
    S = we.forcing.shape[0]
    segs = segments(T, args.steps)
    nseg = len(segs)
    host = {k: torch.from_numpy(np.ascontiguousarray(getattr(we, k))).pin_memory() for k in ("alpha", "n", "ksat", "forcing")}
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, max_fronts=args.max_fronts, chunk_steps=args.chunk, device=dev)
    d_alpha, d_n, d_ksat = (host[k].to(dev) for k in ("alpha", "n", "ksat"))
    if not args.no_balance:
        ens.balance(d_ksat)   # placement of columns on warps by (site, top-layer ksat): lgar_problem.column_order
    outs = ("runoff", "AET")  # per-step series kept in HBM: 2 x T x B x 8 B

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- algorithmic work: closure-call counters of the counting kernel on a sample of whole tiles ----------
    ntiles = (B + 31) // 32
    stride = max(1, int(round(1.0 / max(args.count_fraction, 1e-6))))
    tile_ids = np.arange(0, ntiles, stride)
    cidx = (tile_ids[:, None] * 32 + np.arange(32)[None, :]).reshape(-1)
    cidx = cidx[cidx < B]
    sub = lambda x: np.ascontiguousarray(x[:, cidx])
    ens_c = ColumnEnsemble(theta_r=sub(we.theta_r), theta_e=sub(we.theta_e), thickness=sub(we.thickness), forcing=ens.forcing,
                           site_index=we.site_index[cidx], max_fronts=args.max_fronts, chunk_steps=args.chunk, device=dev)
    res_c, ws_c = forward_raw(ens_c, sub(we.alpha), sub(we.n), sub(we.ksat), outputs=(), per_step=False, counters=True)
    # ... while the GPU counts, rank 0 of a single-GPU run times the CPU port on the first columns of the shard
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        threads = os.cpu_count() or 1
        ncol = min(args.cpu_sample_columns or 48 * threads, B)
        alive_c, dt_c, r_c = port_run(we, np.arange(ncol), T, threads)
        cpu = (alive_c, dt_c, r_c, ncol, threads)
    torch.cuda.synchronize()
    counters = res_c.counters.cpu().numpy()
    alive_sample = int(alive_steps_of(res_c.status.cpu().numpy(), res_c.crash_step.cpu().numpy(), T).sum())
    flop_per_col_step = workloads.algorithmic_flops(counters) / max(alive_sample, 1)
    del res_c, ws_c, ens_c
    torch.cuda.empty_cache()

    # ---- HBM-resident pass, one launch per time segment -------------------------------------------------------
    state = {"res": None, "ws": None}

    pipe = not args.no_pipeline

    def run_segment(i, a, n_, k):
        # consecutive windows are a pipelined sequence (lgar_problem.pipeline_seq): window i+1 starts on the SMs that
        # window i has drained, so the slowest tiles of a window do not idle the GPU at every step boundary
        t0, t1 = segs[i]
        r, state["ws"] = forward_raw(ens, a, n_, k, outputs=outs, workspace=state["ws"], window=(t0, t1), into=state["res"],
                                     pipeline_seq=(i + 1) if pipe else 0)
        state["res"] = r
        return r

    for i in range(args.warmup):
        run_segment(i % nseg, d_alpha, d_n, d_ksat)
    barrier()
    sampler = ClockSampler(local, interval=0.25)
    sampler.start()
    ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(nseg):  # nothing else goes on the stream between the K launches
        run_segment(i, d_alpha, d_n, d_ksat)
    ev1.record()
    barrier()
    total_ms = ev0.elapsed_time(ev1)
    kern_ms = [total_ms]   # the K kernels overlap at their boundaries: only their union is a meaningful duration
    sampler.stop_flag = True
    res = state["res"]
    status = res.status.cpu().numpy()
    crash = res.crash_step.cpu().numpy()
    sums = res.sums.cpu().numpy()
    alive_cols = alive_steps_of(status, crash, T)
    alive_steps = int(alive_cols.sum())
    hist = {lgar_b200.STATUS_NAMES[s]: int((status == s).sum()) for s in np.unique(status)}
    flop_per_pass = flop_per_col_step * alive_steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, segs[-1], outs)

    # ---- parity of the first columns against the oracle results of the cpu_baseline leg ----------------------------
    parity = None
    if cpu:
        _, _, r_c, ncol, _ = cpu
        ITER_CAP = lgar_b200.STATUS_NAMES.index("ITER_CAP")
        FRONT_OVERFLOW = lgar_b200.STATUS_NAMES.index("FRONT_OVERFLOW")
        g_st, o_st = status[:ncol], r_c["status"]
        # ITER_CAP is a limit of the two IMPLEMENTATIONS (the reference would keep iterating): the oracle counts literal
        # iterations, the CUDA root finder crosses long runs in exact jumps and may finish a search the oracle cuts off.
        # FRONT_OVERFLOW is the 16-front capacity of the CUDA kernel (the oracle's lists are unbounded like the
        # reference's; forward_raw(overflow_fallback=True) reruns such columns with 32 fronts).  Columns that end in a
        # capacity status are not comparable beyond that step and are listed separately.
        capped = (g_st == ITER_CAP) | (o_st == ITER_CAP) | (g_st == FRONT_OVERFLOW)
        cmp_ = ~capped
        cr = np.where(crash[:ncol] <= -2, -2 - crash[:ncol], crash[:ncol])
        st_bad = np.nonzero(cmp_ & (o_st != g_st))[0]
        cr_bad = np.nonzero(cmp_ & (o_st != 0) & (o_st == g_st) & (r_c["crash_step"] != cr))[0]
        ok = cmp_ & (o_st == 0) & (g_st == 0)
        g, o = sums[:, :ncol].T[ok], r_c["sums"][ok]
        excess = float(np.max(np.abs(g - o) / (1e-10 + 1e-9 * np.abs(o)), initial=0.0))
        parity = {"columns": int(ncol), "ok_columns": int(ok.sum()), "status_mismatches": int(len(st_bad)),
                  "crash_step_mismatches": int(len(cr_bad)), "max_excess": excess,
                  "capacity_columns_not_compared": int(capped.sum()),
                  "capacity_note": "columns ending in ITER_CAP (either arm) or FRONT_OVERFLOW (CUDA, 16 fronts): library capacity, not reference states",
                  "mismatching_columns": [{"column": int(b), "gpu": [int(g_st[b]), int(cr[b])], "oracle": [int(o_st[b]), int(r_c["crash_step"][b])]}
                                          for b in list(st_bad[:4]) + list(cr_bad[:4])],
                  "what": "full-record sums of all 10 outputs, status and crash step vs the CPU oracle; tolerance 1e-9 rel + 1e-10 abs "
                          "(max_excess <= 1 passes)"}

    # ---- e2e: host tensors in, results out, through the public API, segment by segment ----------------------------
    e2e = None
    if not args.no_e2e:
        seg_len = segs[0][1] - segs[0][0]
        pin = [torch.empty((len(outs), seg_len, B), dtype=torch.float64).pin_memory() for _ in range(2)]
        host_seg = [host["forcing"][:, t0:t1].contiguous().pin_memory() for (t0, t1) in segs]
        copy_stream = torch.cuda.Stream(dev)
        main_stream = torch.cuda.current_stream(dev)
        done_ev = [torch.cuda.Event() for _ in range(2)]
        h2d = d2h = 0

        def e2e_pass(count=False):
            nonlocal h2d, d2h
            a = host["alpha"].to(dev, non_blocking=True)
            n_ = host["n"].to(dev, non_blocking=True)
            k = host["ksat"].to(dev, non_blocking=True)
            if count:
                h2d += 3 * host["alpha"].numel() * 8

            def copy_out(i, r):
                nonlocal d2h
                t0, t1 = segs[i]
                buf = pin[i % 2]
                done_ev[i % 2].synchronize()  # the previous copy into this staging buffer has landed (host may reuse it)
                for q in range(len(outs)):    # contiguous [rows, B] blocks: plain cudaMemcpyAsync
                    buf[q, : t1 - t0].copy_(r.per_step[q, t0:t1], non_blocking=True)
                done_ev[i % 2].record(torch.cuda.current_stream(dev))
                if count:
                    d2h += len(outs) * (t1 - t0) * B * 8

            if args.e2e_interleaved:
                for i, (t0, t1) in enumerate(segs):
                    ens.forcing[:, t0:t1].copy_(host_seg[i], non_blocking=True)
                    r = run_segment(i, a, n_, k)
                    seg_done = torch.cuda.Event()
                    seg_done.record(main_stream)
                    with torch.cuda.stream(copy_stream):
                        copy_stream.wait_event(seg_done)
                        copy_out(i, r)
                    if count:
                        h2d += host_seg[i].numel() * 8
                main_stream.wait_stream(copy_stream)
            else:
                # the whole forcing record is 16 B per site-step: copy it up front, launch the K windows back to back
                # (pipelined), then stream the per-step series out through two bounded pinned staging buffers
                ens.forcing.copy_(host["forcing"], non_blocking=True)
                if count:
                    h2d += host["forcing"].numel() * 8
                for i in range(nseg):
                    r = run_segment(i, a, n_, k)
                for i in range(nseg):
                    copy_out(i, r)
            out = (r.sums.cpu(), r.status.cpu(), r.crash_step.cpu())
            if count:
                d2h += out[0].numel() * 8 + out[1].numel() * 4 + out[2].numel() * 4
            return out

        run_segment(0, d_alpha, d_n, d_ksat)  # touch the path once (allocator, pinned staging)
        barrier()
        t0w = time.perf_counter()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        sums_h, st_h, cr_h = e2e_pass(count=True)
        e1.record()
        barrier()
        e2e_ms = max(e0.elapsed_time(e1), (time.perf_counter() - t0w) * 1e3)
        same = bool(np.array_equal(sums_h.numpy().view(np.int64), sums.view(np.int64)) and np.array_equal(st_h.numpy(), status))
        e2e = (e2e_ms, h2d / nseg, d2h / nseg, same)
        del pin

    # ---- forward + gradient (reverse-mode kernel) over the shard, full record ------------------------------------
    fg = None
    if args.grad_columns > 0:
        from lgar_b200 import lgar_columns
        Bg = min(args.grad_columns, B)
        state["res"] = state["ws"] = res = None
        torch.cuda.empty_cache()
        if Bg == B:
            ens_g, Ag, Ng, Kg = ens, d_alpha, d_n, d_ksat
        else:
            subg = lambda x: np.ascontiguousarray(x[:, :Bg])
            ens_g = ColumnEnsemble(theta_r=subg(we.theta_r), theta_e=subg(we.theta_e), thickness=subg(we.thickness),
                                   forcing=we.forcing, site_index=we.site_index[:Bg], max_fronts=args.max_fronts,
                                   chunk_steps=args.chunk, device=dev)
            Ag, Ng, Kg = (x[:, :Bg].contiguous() for x in (d_alpha, d_n, d_ksat))
            if not args.no_balance:
                ens_g.balance(Kg)
        alive_g = int(alive_cols[:Bg].sum())
        barrier()
        g0 = torch.cuda.Event(enable_timing=True); g1 = torch.cuda.Event(enable_timing=True); gm = torch.cuda.Event(enable_timing=True)
        g0.record()
        A = Ag.clone().requires_grad_(True)
        N_ = Ng.clone().requires_grad_(True)
        Kk = Kg.clone().requires_grad_(True)
        out = lgar_columns(A, N_, Kk, ens_g, outputs=())
        ok = out["status"] == 0
        loss = (out["sums"][0] + out["sums"][2])[ok].mean()   # sum_t runoff + sum_t AET (output indices 0 and 2)
        gm.record()
        loss.backward()
        g1.record()
        barrier()
        gnorm_ok = torch.isfinite(A.grad[:, ok]).all(dim=0) & torch.isfinite(N_.grad[:, ok]).all(dim=0) & torch.isfinite(Kk.grad[:, ok]).all(dim=0)
        fg = (g0.elapsed_time(g1), alive_g, float(gnorm_ok.double().mean()), g0.elapsed_time(gm), float(loss))
        del out, loss, A, N_, Kk

    stats = torch.tensor([total_ms, float(alive_steps), flop_per_pass, e2e[0] if e2e else 0.0,
                          fg[0] if fg else 0.0, float(fg[1]) if fg else 0.0], dtype=torch.float64, device=dev)
    if world > 1:
        mx = stats.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        total_ms_all, e2e_ms_all, fg_ms_all = float(mx[0]), float(mx[3]), float(mx[4])
        alive_all, flop_all, fg_alive_all = float(sm[1]), float(sm[2]), float(sm[5])
    else:
        total_ms_all, e2e_ms_all, fg_ms_all = total_ms, float(stats[3]), float(stats[4])
        alive_all, flop_all, fg_alive_all = float(alive_steps), flop_per_pass, float(stats[5])
    # per-rank pass time, SM clock, power (diagnosis of weak-scaling losses: which rank / GPU was the slow one)
    my_clk = sampler.summary()
    per_rank = torch.tensor([total_ms, float(my_clk["sm_mhz"] or 0.0), float(my_clk["power_w"] or 0.0),
                             1.0 if my_clk["reasons"] else 0.0, float(alive_steps), fg[0] if fg else 0.0, flop_per_pass],
                            dtype=torch.float64, device=dev)
    if world > 1:
        gathered = [torch.zeros_like(per_rank) for _ in range(world)]
        dist.all_gather(gathered, per_rank)
    else:
        gathered = [per_rank]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    ms_per_step = total_ms_all / nseg
    value = alive_all / (total_ms_all * 1e-3)
    fp64_peak = _capi.lib().lgar_measure_fp64_flops(8192)
    kern_s = float(np.sum(kern_ms)) * 1e-3           # rank 0's kernels over the pass
    achieved = flop_per_pass / kern_s
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    out_bytes = len(outs) * T * B * 8 + T * 16 * S
    traffic_note = None
    try:  # dram bytes per launch from the committed ncu capture of this kernel (profiles/), scaled per column-step
        tr = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        traffic = tr["dram_bytes_per_column_step"] * alive_steps / nseg
        traffic_note = tr.get("source")
    except Exception:
        traffic = None
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": nseg, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(args), "columns_per_gpu": B, "forcing_steps": T,
                   "step": f"one time segment of {segs[0][1] - segs[0][0]} forcing rows over the whole shard; the {nseg} timed steps are "
                           "one pass over the full record (resume launches, bit-identical to one launch)"
                           + ("; consecutive windows are pipelined with programmatic dependent launch" if pipe else ""),
                   "ok_fraction": float((status == 0).mean()), "status_histogram": hist,
                   "status_note": "non-OK columns are the reference's exceptions at the same step (it aborts the run); "
                                  "FRONT_OVERFLOW (>16 fronts) and ITER_CAP (a root finder above 1e6 iterations, where the "
                                  "reference keeps looping for hours) are capacity limits of this library, not reference states",
                   "alive_column_steps_per_gpu": alive_steps, "max_fronts": args.max_fronts, "chunk_steps": args.chunk,
                   "placement": "identity" if args.no_balance else "columns sorted by (site, top-layer ksat) (ColumnEnsemble.balance)",
                   "l2": "working set per step (per-step outputs %d x %d x B x 8 B = %.2f GB) exceeds the 126 MB L2; no flush needed"
                         % (len(outs), segs[0][1] - segs[0][0], len(outs) * (segs[0][1] - segs[0][0]) * B * 8 / 1e9)},
        "gpu_launches": nseg,
        "clocks": my_clk,
        "per_rank": {"pass_ms": [float(g[0]) for g in gathered], "sm_mhz": [float(g[1]) for g in gathered],
                     "power_w": [float(g[2]) for g in gathered], "throttle_reason_seen": [bool(g[3] > 0) for g in gathered],
                     "alive_column_steps": [float(g[4]) for g in gathered], "fwd_grad_ms": [float(g[5]) for g in gathered],
                     # algorithmic flop of each rank's shard (its own counting pass) / its own pass time: equal rates with
                     # unequal pass times = the shards differ in work, not the GPUs in speed
                     "achieved_tflops": [float(g[6]) / (float(g[0]) * 1e-3) / 1e12 for g in gathered]},
        "roofline": {"bound": "fp64", "achieved": achieved / 1e12, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
                     "frac": achieved / fp64_peak if fp64_peak else None, "traffic": traffic, "traffic_source": traffic_note,
                     "peak_source": "in-run DFMA probe (lgar_measure_fp64_flops); MEASURED_PEAKS.json has no FP64 entry",
                     "flop_per_column_step": flop_per_col_step,
                     "flop_source": f"closure-call counters of the counting kernel on every {stride}th tile of the shard "
                                    f"({len(cidx)} columns, full record) x SURVEY 8d weights (pow = 125 flop)",
                     "executed_frac_note": "this library's pow executes ~100 FP64 flop, not 125: see profiles/ for the executed-flop fraction (ncu)",
                     "hbm": {"algorithmic_bytes_per_pass": out_bytes, "achieved_gbs": out_bytes / kern_s / 1e9,
                             "peak_gbs": hbm_peak, "frac": out_bytes / kern_s / 1e9 / hbm_peak}},
        "wall_s": None,
    }
    if parity:
        line["parity"] = parity
    if fg:
        fg_val = fg_alive_all / (fg_ms_all * 1e-3)
        fg_flop = 2.0 * flop_per_col_step * fg[1]   # forward + taped recompute of every sub-step (adjoint sweep not counted)
        line["fwd_grad"] = {"value": fg_val, "unit": UNIT, "columns_per_gpu": min(args.grad_columns, B), "forcing_steps": T,
                            "ms": fg_ms_all, "forward_ms": fg[3], "loss": fg[4],
                            "what": "lgar_forward(keep checkpoints) + lgar_backward through torch.autograd over the whole shard and "
                                    "record, loss = mean over OK columns of sum_t (runoff + AET)",
                            "finite_grad_fraction_ok_columns": fg[2],
                            "roofline": {"achieved": fg_flop / (fg[0] * 1e-3) / 1e12, "peak": fp64_peak / 1e12, "unit": "TFLOP/s",
                                         "frac": fg_flop / (fg[0] * 1e-3) / fp64_peak if fp64_peak else None,
                                         "flop": "2 x forward algorithmic flop (forward + taped recompute); adjoint sweep not counted"}}
    if e2e:
        line["e2e"] = {"value": alive_all / (e2e_ms_all * 1e-3), "unit": UNIT, "h2d_bytes_per_step": e2e[1],
                       "d2h_bytes_per_step": e2e[2], "ms_per_step": e2e_ms_all / nseg, "bit_identical_to_resident_pass": e2e[3],
                       "what": ("forward_raw per segment: pinned forcing segment H2D (+ parameters at step 0), launch, D2H of the segment's "
                                "per-step runoff and AET on a copy stream, sums/status/crash_step at the end") if args.e2e_interleaved else
                               ("pinned parameters + forcing record H2D, the K window launches back to back (pipelined), D2H of the per-step "
                                "runoff and AET series through two pinned staging buffers, then sums/status/crash_step; bytes are per step "
                                "(= total / K)")}
    if cpu:
        alive_c, dt_c, _, ncol, threads = cpu
        line["cpu_baseline"] = {"value": alive_c / dt_c, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"columns 0..{ncol - 1} x {T} steps of the same ensemble (alive column-steps), {dt_c:.1f} s, "
                                          "C++ restatement of the reference; the Python reference itself is timed by --impl reference"}
    line["wall_s"] = time.perf_counter() - t_start
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
