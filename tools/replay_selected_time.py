"""Cost of select-then-replay on one GPU: phase 1 = all chains with no sample store (SER_STORE_NONE), phase 2 = the k chosen
chains re-simulated alone (ser_run_create_chains) with the pair-order counts and posterior sums accumulating through a window
of W samples (ser_run_accumulate), at the reference's 1000 + 1000 schedule.

    python tools/replay_selected_time.py [--out FILE.json] [--windows 16,64,256] [--quick]

Per case and window: phase-2 wall time (host clock around the launches and a final synchronise), the CUDA-event time of the
sweep launches alone, and the summed kernel time of the accumulation kernels (torch.profiler, in a separate profiled pass
so the wall time is taken without tracing; that pass only advances the run, so every launch of a summary kernel in it is an
accumulation).  Device memory of each phase = memory in use (cudaMemGetInfo) after the phase's
run is created, initialised and has taken a sample, minus what was in use before; the library's pool keeps no freed blocks
(SER_POOL_KEEP_MB=0).  Phase 1 runs only 1 + 1 calls: it is here for its memory and to choose the chains, whose phase-2
cost does not depend on which chains they are.  --quick shortens everything to a rehearsal.
"""
import argparse
import json
import os
import subprocess
import sys
import time

os.environ["SER_POOL_KEEP_MB"] = "0"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import seriation_b200 as S  # noqa: E402
from tools.datasets import load_hex_dataset  # noqa: E402

ACC_KERNELS = ("ser_po_kernel", "ser_posterior_kernel")


def used_bytes(torch):
    torch.cuda.synchronize()
    free, total = torch.cuda.mem_get_info(0)
    return total - free


def phase2(torch, ds, ids, burn, samples, window, profile):
    run = S.Run(ds, 0, seed=20060206, store=S.STORE_PI, max_samples=window, chain_ids=ids).init().accumulate(po=True, sums=True)
    run.sync()
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
    per = {}
    for e in p.key_averages():
        t = getattr(e, "self_device_time_total", None)
        t = e.self_cuda_time_total if t is None else t
        if t > 0:
            per[e.key] = (t / 1e3, e.count)
    acc = {k: v for k, v in per.items() if any(a in k for a in ACC_KERNELS)}
    sweep = {k: v for k, v in per.items() if "ser_sweep_kernel" in k}
    return dict(acc_kernel_ms=sum(v[0] for v in acc.values()), acc_launches=sum(v[1] for v in acc.values()),
                profiled_sweep_kernel_ms=sum(v[0] for v in sweep.values()), kernels={k: v[0] for k, v in per.items()})


def case(torch, label, ds, n1, k, burn, samples, windows):
    N = ds.N
    base = used_bytes(torch)
    run = S.Run(ds, n1, seed=20060206, store=S.STORE_NONE, max_samples=samples).init().advance(1, False).advance(1, True)
    p1_bytes = used_bytes(torch) - base
    chosen, _, _ = S.select_chains(run.chain_stats()["e_negloglik"], k)
    run.close()
    ids = [int(c) for c in chosen]
    out = dict(case=label, N=N, M=ds.M, phase1_chains=n1, k=len(ids), chosen=ids, burn=burn, samples=samples,
               phase1_device_bytes=p1_bytes, one_shot_pi_store_bytes=n1 * samples * N * 2, windows=[])
    for W in windows:
        base = used_bytes(torch)
        probe = S.Run(ds, 0, seed=20060206, store=S.STORE_PI, max_samples=W, chain_ids=ids).init().accumulate(po=True, sums=True)
        probe.advance(1, True)
        p2_bytes = used_bytes(torch) - base
        probe.close()
        timed = phase2(torch, ds, ids, burn, samples, W, profile=False)
        profiled = phase2(torch, ds, ids, burn, samples, W, profile=True)
        row = dict(window=W, phase2_device_bytes=p2_bytes, **timed, **profiled)
        row["acc_share_of_sweep"] = row["acc_kernel_ms"] / row["sweep_ms"] if row["sweep_ms"] else None
        out["windows"].append(row)
        print(json.dumps({k: v for k, v in row.items() if k != "kernels"}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the full results (incl. per-kernel times) as JSON here")
    ap.add_argument("--windows", default="16,64,256")
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("replay_selected_time: needs a CUDA device")
    windows = [int(w) for w in a.windows.split(",")]
    burn = samples = 20 if a.quick else 1000
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    X, hard = load_hex_dataset("g2s2")
    res = dict(gpu=gpu, cases=[])
    res["cases"].append(case(torch, "g2s2 k=4", S.Dataset.from_bits(X, hard), 1024 if a.quick else 65536, 4, burn, samples, windows))
    res["cases"].append(case(torch, "synthetic 1024x4096 (config 5) k=2", S.Dataset.synthetic(1024, 4096, 16),
                             512 if a.quick else 65536, 2, burn, samples, windows))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print("gpu:", gpu)


if __name__ == "__main__":
    main()
