"""Cost of the rank-normalised diagnostics on one GPU: device time of the kernels of one ser_run_rank_diagnostics call and its
wall time.

    python tools/rank_diagnostics_time.py [--out FILE.json] [--reps R] [--quick]

Cases (T = 1000 stored samples per chain, every quantity: -loglik, exp(c), exp(d) and pi of every site):
  g2s2, k = 4 chosen chains;  the 1024 x 4096 synthetic matrix (BASELINE.json config 5), k = 2.
Each run samples T calls (config 5: one sweep per call, as in tools/diagnostics_time.py), then ser_run_rank_diagnostics is called
twice to warm up and R times under torch.profiler with CUDA activities: per kernel name (ser_rank_*, and CUB's radix sort as
"cub sort"), the device time over R.  The wall time (host clock around the call, which reads the chains' sample counts, copies
`out` in and out and synchronises) is taken in the same loop.  The card's name and power limit are read in the same process.
--quick shrinks the cases to a rehearsal.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import seriation_b200 as S  # noqa: E402
from tools.datasets import load_hex_dataset  # noqa: E402


def case(label, ds, n, chosen, T, spc, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    run = S.Run(ds, n, seed=20060206, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T).init().advance(T, True).sync()
    chosen = np.asarray(chosen, np.int32)
    for _ in range(2):
        rd = run.rank_diagnostics(chosen)
    wall = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            t0 = time.perf_counter()
            run.rank_diagnostics(chosen)
            wall.append(time.perf_counter() - t0)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        name = "cub sort" if "cub" in e.key.lower() else e.key if "ser_rank" in e.key else None
        if name is None or "Memcpy" in e.key or "Memset" in e.key:
            continue
        t = getattr(e, "self_device_time_total", None)
        kernels[name] = kernels.get(name, 0.0) + (e.self_cuda_time_total if t is None else t) / reps / 1e3
    if not any("ser_rank_ess_kernel" in k for k in kernels):
        sys.exit("rank_diagnostics_time: the profiler saw no ser_rank_ess_kernel launch")
    Q = 3 + ds.N
    row = dict(case=label, N=ds.N, M=ds.M, k=int(chosen.size), T=T, sweeps_per_call=spc, quantities=Q,
               kernel_ms=sum(kernels.values()), kernels_ms=kernels, wall_ms=[1e3 * w for w in wall],
               max_rhat=float(np.nanmax(rd["rhat"][np.isfinite(rd["rhat"])])), min_ess_bulk=float(np.nanmin(rd["ess_bulk"])))
    print(json.dumps(row), flush=True)
    run.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the results as JSON here")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("rank_diagnostics_time: needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    T = 100 if a.quick else 1000
    res = dict(gpu=gpu, cases=[
        case("g2s2", S.Dataset.from_bits(*load_hex_dataset("g2s2")), 16, [1, 5, 9, 13], T, 10, a.reps),
        case("synthetic 1024x4096 (config 5)", S.Dataset.synthetic(1024, 4096, 16), 2, [0, 1], T, 1, a.reps),
    ])
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
