"""Cost of the diversity curves on one GPU.

    python tools/diversity_time.py [--out FILE.json] [--windows 16,64,256] [--reps R] [--quick]

One-shot (ser_run_diversity over a store that holds every sample, all four outputs): g2s2 with k = 4 chains and the 1024 x 4096
synthetic matrix (BASELINE.json config 5, a large-shape kernel run) with k = 2, T = 1000 samples per chain.  The call is made twice to
warm up and R times under torch.profiler with CUDA activities: kernel time = device time of ser_div_curve_kernel (stage 1) and
ser_div_hist_kernel (stage 2) over R; wall time = host clock around the call (which copies the four [k][N][M+1] slabs back and
synchronises), taken in the same loop.

Phase 2 of select-then-replay (the k chosen chains of a 65 536-chain phase 1 re-simulated alone at 1000 + 1000 calls through a window of
W samples), without the diversity curves (SER_STORE_PI, SER_ACC_PO | SER_ACC_SUMS, as replay_selected_time.py) and with them
(SER_STORE_FULL, + SER_ACC_DIV): wall time, CUDA-event time of the sweep launches, and in a separate profiled pass the summed device time
of the accumulation kernels: the summary kernels serve both paths, so in a pass that only advances the run every launch of them is an
accumulation.  The card's name and power limit are read in the same process.  --quick shrinks everything to a rehearsal.
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
from tools.marginals_time import kernel_ms  # noqa: E402

ONE_SHOT = ("ser_div_curve_kernel", "ser_div_hist_kernel")
ACC = ("ser_po_kernel", "ser_posterior_kernel") + ONE_SHOT


def one_shot(label, ds, n, chosen, T, spc, reps):
    from torch.profiler import ProfilerActivity, profile
    run = S.Run(ds, n, seed=20060206, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T).init().advance(T, True).sync()
    path = run.kernel_path()
    for _ in range(2):
        run.diversity(chosen)
    wall = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            t0 = time.perf_counter()
            run.diversity(chosen)
            wall.append(time.perf_counter() - t0)
    per = kernel_ms(prof, ONE_SHOT)
    run.close()
    k = len(chosen)
    row = dict(case=label, N=ds.N, M=ds.M, k=k, T=T, sweep_kernel_path=path, reps=reps,
               kernel_ms_per_call=sum(per.values()) / reps, kernels_ms_per_call={name: v / reps for name, v in per.items()},
               out_bytes=16 * k * ds.N * (ds.M + 1), wall_s_min=min(wall), wall_s_median=float(np.median(wall)))
    print(json.dumps(row), flush=True)
    return row


def phase2(ds, ids, burn, samples, window, div, profile):
    store = S.STORE_FULL if div else S.STORE_PI
    run = S.Run(ds, 0, seed=20060206, store=store, max_samples=window, chain_ids=ids).init()
    run.accumulate(po=True, sums=True, diversity=div).sync()
    run.sweep_time(reset=True)
    if not profile:
        t0 = time.perf_counter()
        run.advance(burn, False).advance(samples, True).sync()
        wall = time.perf_counter() - t0
        sweep_ms, launches = run.sweep_time(reset=True)
        run.close()
        return dict(wall_s=wall, sweep_ms=sweep_ms, sweep_launches=launches)
    from torch.profiler import ProfilerActivity, profile as prof
    with prof(activities=[ProfilerActivity.CUDA]) as p:
        run.advance(burn, False).advance(samples, True).sync()
    run.close()
    per = kernel_ms(p, ACC)
    return dict(acc_kernel_ms=sum(per.values()), acc_kernels_ms=per)


def replay_case(label, ds, n1, k, burn, samples, windows):
    run = S.Run(ds, n1, seed=20060206, store=S.STORE_NONE, max_samples=samples).init().advance(1, False).advance(1, True)
    chosen, _, _ = S.select_chains(run.chain_stats()["e_negloglik"], k)
    run.close()
    ids = [int(c) for c in chosen]
    rows = []
    for W in windows:
        for div in (False, True):
            row = dict(case=label, window=W, diversity=div, k=len(ids), burn=burn, samples=samples,
                       **phase2(ds, ids, burn, samples, W, div, profile=False), **phase2(ds, ids, burn, samples, W, div, profile=True))
            row["acc_share_of_wall"] = row["acc_kernel_ms"] / (row["wall_s"] * 1e3)
            rows.append(row)
            print(json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the results as JSON here")
    ap.add_argument("--windows", default="16,64,256")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("diversity_time: needs a CUDA device")
    windows = [int(w) for w in a.windows.split(",")]
    T = burn = samples = 20 if a.quick else 1000
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("gpu:", gpu, flush=True)
    g2s2 = S.Dataset.from_bits(*load_hex_dataset("g2s2"))
    syn = S.Dataset.synthetic(1024, 4096, 16)
    res = dict(gpu=gpu, one_shot=[], phase2=[])
    res["one_shot"].append(one_shot("g2s2 k=4", g2s2, 4, [0, 1, 2, 3], T, 10, a.reps))
    res["one_shot"].append(one_shot("synthetic 1024x4096 (config 5) k=2", syn, 2, [0, 1], T, 1, a.reps))
    res["phase2"] += replay_case("g2s2 k=4", g2s2, 1024 if a.quick else 65536, 4, burn, samples, windows)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
