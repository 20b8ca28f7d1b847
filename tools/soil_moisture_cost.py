"""Cost of the soil-moisture outputs on the C4 shard (one GPU): 125,000 columns x 8760 h of
workloads.synthetic_sites_ensemble, balanced placement, the record advanced in the same pipelined windows bench.py
times (lgar_problem.pipeline_seq), timed with CUDA events around work that ends in a synchronise.  Arms, alternated
round by round in one process:

  1 fwd           forward, runoff and AET stored per step (bench.py's outputs), no soil-moisture output
  2 fwd+sm        arm 1 plus theta at 5 depths and the water of the 3 layers stored for every step of the year
                  (skipped with a note when the device lacks the memory for them)
  3 fwd+sm_last   arm 1 plus the soil-moisture outputs requested for the last window only
  4 grad          forward + gradient, loss = sum runoff + sum AET + final volume, on --grad-columns columns
  5 grad+sm       arm 4 plus an MSE on theta at the 5 depths

Prints one JSON line per arm and round, with the GPU name and power limit read in the same process.
Usage: python tools/soil_moisture_cost.py [--rounds 2] [--columns 125000] [--grad-columns 12500] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

DEPTHS = (5.0, 10.0, 20.0, 50.0, 100.0)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--columns", type=int, default=125_000)
    ap.add_argument("--nsteps", type=int, default=8760)
    ap.add_argument("--steps", type=int, default=20, help="pipelined windows per pass (bench.py --steps)")
    ap.add_argument("--grad-columns", type=int, default=12_500)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "the cost of the outputs is a GPU figure: no device, no measurement"
    import bench
    from lgar_b200 import ColumnEnsemble, forward_raw, lgar_columns, workloads
    dev = torch.device("cuda", 0)
    B, T = args.columns, args.nsteps
    we = workloads.synthetic_sites_ensemble(B=B, T=T, shared_sites=True)
    segs = bench.segments(T, args.steps)
    ens = ColumnEnsemble(theta_r=we.theta_r, theta_e=we.theta_e, thickness=we.thickness, forcing=we.forcing,
                         site_index=we.site_index, moisture_depths=DEPTHS, device=dev)
    a, n, k = (torch.tensor(getattr(we, x), device=dev) for x in ("alpha", "n", "ksat"))
    ens.balance(k)
    info = gpu_info()
    out_f = open(args.out, "a") if args.out else None

    def emit(rec):
        rec.update(gpu=info, columns=rec.get("columns", B), steps=T, windows=len(segs), depths=list(DEPTHS))
        line = json.dumps(rec)
        print(line, flush=True)
        if out_f:
            out_f.write(line + "\n")
            out_f.flush()

    def forward_pass(sm):
        """sm: None (no soil moisture), 'all' (every window) or 'last' (last window only)."""
        res, ws = None, None
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i, (t0, t1) in enumerate(segs):
            want = sm == "all" or (sm == "last" and i == len(segs) - 1)
            res, ws = forward_raw(ens, a, n, k, outputs=("runoff", "AET"), workspace=ws, window=(t0, t1), into=res,
                                  pipeline_seq=i + 1, moisture=want, layer_water=want)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        ok = int((res.status == 0).sum())
        del res, ws
        torch.cuda.empty_cache()
        return ms, ok

    Bg = min(args.grad_columns, B)
    cols = torch.arange(Bg, device=dev)
    sub = lambda x: x[:, cols].contiguous()
    ens_g = ColumnEnsemble(theta_r=sub(ens.theta_r), theta_e=sub(ens.theta_e), thickness=sub(ens.thickness),
                           forcing=ens.forcing, site_index=ens.site_index[cols], moisture_depths=DEPTHS, device=dev)
    ens_g.balance(sub(k))

    def grad_pass(sm):
        A, N, K = (sub(x).clone().requires_grad_(True) for x in (a, n, k))
        torch.cuda.synchronize()
        t = time.perf_counter()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = lgar_columns(A, N, K, ens_g, outputs=("moisture",) if sm else ())
        ok = out["status"] == 0
        loss = (out["sums"][0] + out["sums"][2] + out["sums"][4])[ok].sum()
        if sm:
            loss = loss + ((out["moisture"][:, :, ok] - 0.3) ** 2).sum()
        loss.backward()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        wall = (time.perf_counter() - t) * 1e3
        okc = int(ok.sum())
        del out, loss, A, N, K
        torch.cuda.empty_cache()
        return ms, wall, okc

    # arm 2 keeps 5 + 3 doubles per column-step for the whole year next to bench.py's two series
    need_sm = (len(DEPTHS) + ens.num_layers) * T * B * 8
    forward_pass(None)   # warm-up: module load, workspace, first launches of every instantiation used
    forward_pass("last")
    grad_pass(True)
    for r in range(args.rounds):
        ms, ok = forward_pass(None)
        emit(dict(round=r, arm=1, what="forward, no soil-moisture output", ms=ms, ok_columns=ok))
        free, _ = torch.cuda.mem_get_info(dev)
        if free > need_sm * 1.2 + 4 * T * B * 8:
            ms, ok = forward_pass("all")
            emit(dict(round=r, arm=2, what="forward, theta at 5 depths + 3 layer waters stored every step",
                      ms=ms, ok_columns=ok, extra_bytes=need_sm, extra_bytes_per_column_step=need_sm / (T * B)))
        else:
            emit(dict(round=r, arm=2, what="not run: device memory", free_bytes=free, needed_bytes=need_sm))
        ms, ok = forward_pass("last")
        emit(dict(round=r, arm=3, what="forward, soil-moisture outputs requested for the last window only", ms=ms,
                  ok_columns=ok))
        for arm, sm in ((4, False), (5, True)):
            ms, wall, ok = grad_pass(sm)
            emit(dict(round=r, arm=arm, columns=Bg,
                      what="forward+gradient, sum runoff + sum AET + final volume" + (" + MSE theta(5 depths)" if sm else ""),
                      ms=ms, wall_ms=wall, ok_columns=ok))


if __name__ == "__main__":
    main()
