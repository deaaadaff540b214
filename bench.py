#!/usr/bin/env python
"""bench.py -- aggregate MCMC sweeps/s across chains (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py ... --dump-outputs DIR                   (+ the last timed step's results as DIR/*.npy)
    python bench.py --impl reference --steps K --warmup W    (the reference's CPU path)

Workload = BASELINE.json config 4: g2s2 (526 x 296, the largest NOW subset), 16 384 chains IN TOTAL, sharded over the
N ranks by global chain id ("scaling": "strong"; no data-path traffic).  One *step* = one whole job over the batch:
randomised start (init kernel), burn-in calls + sampling calls in one persistent launch with thinned-sample
streaming, and the cross-chain step -- E[-logL] per chain -> all-gather -> within-one-sigma selection -> pair-order
counts of the selected chains -> all-reduce -- enqueued on one stream by the C library (NCCL through ser_comm_* at
N > 1; torch.distributed only broadcasts the communicator id).

Prints ONE JSON line (rank 0).  `value` times the job with all inputs resident in HBM; `e2e` times the same job
through the host-buffer C ABI (dataset upload, run creation, results copied back to host).  `roofline` reports
the sweep kernel (CUDA events around every sweep launch of the timed region) against the SM-local FP64 ceiling
measured live by ser_microbench (the path is neither HBM- nor tensor-bound, SURVEY.md section 8d);
`cpu_baseline` times the unmodified reference (oracle/_ref) on the host cores.  `also` carries BASELINE.json
config 5 as a full line at every N (65 536 chains of the 1024 x 4096 synthetic matrix in total) and, at N = 1,
the reference's actual regime (1000 burn-in calls, then 1000 sampling calls with 1000 stored samples).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

# algorithmic work per sweep (SURVEY.md section 8d closed forms): canonical cells C, smem bytes B = C/8,
# fp64 candidate weights F = M(N+2) -> 10 F flops, HBM bytes per thinned sample
ALGO = {
    "g10s10": dict(N=124, M=139, C=74967, B=9371, F=17514, hbm_sample=828, k=8),
    "g10s2": dict(N=501, M=139, C=301352, B=37669, F=69917, hbm_sample=1582, k=2),
    "g5s5": dict(N=273, M=202, C=238360, B=29795, F=55550, hbm_sample=1378, k=2),
    "g2s2": dict(N=526, M=296, C=673301, B=84163, F=156288, hbm_sample=2260, k=4),
    "synthetic": dict(N=1024, M=4096, C=18149376, B=2268672, F=4202496, hbm_sample=18456, k=2),
}
TOTAL_CHAINS = {"g10s10": 16384, "g10s2": 16384, "g5s5": 16384, "g2s2": 16384, "synthetic": 65536}  # BASELINE.json configs 4, 5
METRIC = "mcmc_sweeps_per_s_aggregate"
UNIT = "sweeps/s"
# DRAM traffic of the sweep kernels from the committed `ncu --set full` captures (profiles/r02/README.md).
# ser_sweep_kernel: dram__bytes_read.sum + dram__bytes_write.sum = 103.29 MB + 167.47 MB over the 8 192 work items of the profiled
# launch (4 096 chains x 2 one-call items) = 33.05 KB per work item -- the chain state incl. its bit columns going through HBM at an
# item boundary; the thinned samples add 2 N bytes each.  ser_sweep_kernel_big (warp batches): 1.263 GB + 1.210 GB over 2 960 chain-sweeps.
NCU_DRAM = {"g2s2": dict(per_item=(102.342656e6 + 163.281920e6) / 8192, src="profiles/r02/sweep_r02_v3_ncu_raw_selected.txt"),
            "synthetic": dict(per_sweep=(1.263233e9 + 1.209718e9) / 2960, src="profiles/r02/sweep_big_r02_warpbatch_ncu_raw_selected.txt")}


def workload_name(dataset):
    a = ALGO[dataset]
    return "%s %dx%d, %d chains in total, thin 10 (BASELINE.json config %d)" % (dataset, a["N"], a["M"], TOTAL_CHAINS[dataset],
                                                                              5 if dataset == "synthetic" else 4)


def load_dataset(name):
    """(X, hard): a NOW subset from the committed fixtures, or the deterministic 1024 x 4096 synthetic
    matrix of BASELINE.json config 5 (generator: ser_dataset_synthetic, DESIGN.md)"""
    if name == "synthetic":
        import seriation_b200 as S
        return S.Dataset.synthetic(1024, 4096, 16).arrays()
    from tools.datasets import load_hex_dataset
    return load_hex_dataset(name)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dataset", default="g2s2", choices=sorted(ALGO))
    ap.add_argument("--chains", type=int, default=0, help="chains IN TOTAL over all GPUs (0: 16384; synthetic: 65536)")
    ap.add_argument("--burn-calls", type=int, default=0, help="0: 5 (synthetic: 1)")
    ap.add_argument("--sample-calls", type=int, default=0, help="0: 5 (synthetic: 1)")
    ap.add_argument("--no-synthetic", action="store_true", help="skip the config-5 line under `also`")
    ap.add_argument("--no-stationary", action="store_true", help="skip the 1000 + 1000 call regime under `also`")
    ap.add_argument("--stationary-chains", type=int, default=4096)
    ap.add_argument("--cpu-calls", type=int, default=0, help="mcmc_sample() calls per CPU process (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy "
                    "(float64; rank 0: the global cross-chain result and its own shard's per-chain arrays)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


# ------------------------------------------------------------------ CPU reference arm
def cpu_reference_run(dataset, calls, procs):
    """`procs` concurrent processes of the reference sampler (script.py's Pool, :60-62), each doing
    `calls` mcmc_sample() calls (= 10 sweeps each) on `dataset`.  Returns (sweeps/s aggregate, kind)."""
    from oracle import oracle as O
    from tools.datasets import write_txt
    X, hard = load_dataset(dataset)
    ref_bin = O.REF_BIN + ("_big" if X.shape[1] > 900 else "")  # rows > 1999 chars need the MAXS-patched build
    if O.ref_available() and os.access(ref_bin, os.X_OK):
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, dataset + ".txt")
            write_txt(path, X, hard)
            t0 = time.perf_counter()
            ps = [subprocess.Popen([ref_bin, "bench", path, str(calls)], env=dict(os.environ, GSL_RNG_SEED=str(i + 1)),
                                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL) for i in range(procs)]
            rcs = [p.wait() for p in ps]
            dt = time.perf_counter() - t0
        if any(rcs):
            raise RuntimeError("reference binary failed: %r" % rcs)
        return procs * calls * 10 / dt, "reference"
    # no prebuilt reference binary: time the restatement (one process per core)
    code = ("import sys; sys.dont_write_bytecode = True; sys.path.insert(0, %r); from oracle import oracle as O; import bench;"
            "X,h=bench.load_dataset(%r); o=O.Oracle(X,h).source_mt(int(sys.argv[1])); o.randomize();"
            "[o.sample() for _ in range(%d)]" % (ROOT, dataset, calls))
    O.build()
    t0 = time.perf_counter()
    ps = [subprocess.Popen([sys.executable, "-c", code, str(i + 1)]) for i in range(procs)]
    rcs = [p.wait() for p in ps]
    dt = time.perf_counter() - t0
    if any(rcs):
        raise RuntimeError("oracle port failed: %r" % rcs)
    return procs * calls * 10 / dt, "port"


def auto_cpu_calls(dataset):
    # ~10 s of CPU work per process: the survey measured 24-26 ns per canonical cell
    per_sweep = ALGO[dataset]["C"] * 25e-9
    return max(1, int(10.0 / (per_sweep * 10)))


def cpu_sample_text(procs, calls, dataset):
    return ("%d concurrent processes (os.cpu_count(); script.py's Pool uses 8) x %d mcmc_sample() calls = %d sweeps each of %s, "
            "from mcmc_randomize's start; unmodified mcmc.c -O2 behind the GSL-API shim; the chain_data.csv / exp_data.csv "
            "output of the reference's main() is omitted (favours the CPU)" % (procs, calls, calls * 10, dataset))


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    procs = os.cpu_count() or 1
    calls = args.cpu_calls or auto_cpu_calls(args.dataset)
    for _ in range(args.warmup):
        cpu_reference_run(args.dataset, max(1, calls // 8), procs)
    t0 = time.perf_counter()
    vals = [cpu_reference_run(args.dataset, calls, procs) for _ in range(args.steps)]
    dt = time.perf_counter() - t0
    value = sum(v for v, _ in vals) / len(vals)
    kind = vals[0][1]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "NOW subset %s (committed fixture of the reference's Dataset/)" % args.dataset,
        "config": {"workload": workload_name(args.dataset), "arm": "reference C sampler (mcmc.c, -O2, GSL-API shim) on the host cores, "
                   "a bounded sample of the workload per step", "sweeps_per_step": procs * calls * 10},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": kind, "sample": cpu_sample_text(procs, calls, args.dataset)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------ the B200 arm
class Job:
    """one workload (dataset, total chains, calls) on this rank's shard"""

    def __init__(self, S, dataset, total, burn, samp, k, rank, world, local, comm):
        self.S, self.dataset, self.burn, self.samp, self.k = S, dataset, burn, samp, k
        self.rank, self.world, self.local, self.comm = rank, world, local, comm
        assert total % world == 0, "the chains must divide over the ranks"
        self.n_local, self.total = total // world, total
        self.X, self.hard = load_dataset(dataset)
        self.N, self.M = self.X.shape
        self.sweeps_per_step = total * (burn + samp) * 10

    def make_run(self, ds=None):
        S = self.S
        ds = ds or S.Dataset.from_bits(self.X, self.hard)
        return S.Run(ds, self.n_local, mode=S.MODE_FREE, seed=20060206, chain_offset=self.rank * self.n_local, store=S.STORE_PI,
                     max_samples=self.samp, device=self.local)

    def step_resident(self, run):
        """inputs resident: the run object (dataset bits, state buffers) already lives in HBM; results stay there"""
        run.init().advance_both(self.burn, self.samp).cross_chain_async(self.k, self.comm)

    def step_e2e(self):
        """host buffers in, host results out, through the C ABI"""
        S = self.S
        run = self.make_run(S.Dataset.from_bits(self.X, self.hard))           # host -> library (bit-packed on upload)
        run.init().advance_both(self.burn, self.samp)
        res = run.cross_chain(self.k, self.comm)                                 # D2H: chosen ids, k x N x N counts
        po = S.po_finalize(res["counts"][:max(1, len(res["chosen"]))], self.k) if len(res["chosen"]) else None
        run.close()
        return 0.0 if po is None else float(po[0, 1])

    def bytes_per_step(self):
        h2d = int(self.N * ((self.M + 31) // 32) * 4 + self.N + 12 * self.M)
        d2h = int(self.k * self.N * self.N * 4 + self.k * 4 + 24)
        return h2d, d2h


def _seeded_rows(n, cap):
    """all of range(n), or a fixed sorted sample of `cap` of them"""
    import numpy as np
    return np.arange(n) if n <= cap else np.sort(np.random.default_rng(20060206).choice(n, cap, replace=False))


def dump_outputs(out_dir, job, run):
    """What a caller of the timed path receives from its last step, so that two builds can be compared output for output (the
    inputs -- dataset, seed, chain ids -- are fixed by the arguments): the cross-chain result (chosen global chain ids, the
    E[-logL] minimum and sigma, the chosen chains' pair-order counts), E[-logL], E[c], E[d] of every chain of this rank, and
    the final state and stored pi samples of a fixed sample of 64 chains.  float64 holds every integer here exactly; per-chain
    arrays beyond 262 144 chains are sampled the same way, which keeps the dump under 64 MB for every dataset."""
    import numpy as np
    res = run.cross_chain_result()
    stats = run.chain_stats()
    rows = _seeded_rows(job.n_local, 1 << 18)
    some = _seeded_rows(job.n_local, 64)
    states = [run.state(int(i)) for i in some]
    out = {"chosen": res["chosen"], "min_sigma": [res["min"], res["sigma"]], "po_counts": res["counts"][:len(res["chosen"])],
           "chain_ids": rows + job.rank * job.n_local, "e_negloglik": stats["e_negloglik"][rows], "e_c": stats["e_c"][rows],
           "e_d": stats["e_d"][rows], "sample_chain_ids": some + job.rank * job.n_local,
           "sample_pi_history": np.stack([run.fetch_samples(int(i), full=False)["pi"] for i in some])}
    for k in ("a", "b", "pi", "c", "d", "loglik"):
        out["sample_" + k] = np.stack([s[k] for s in states])
    os.makedirs(out_dir, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(v, dtype=np.float64))


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import seriation_b200 as S

    # stdout carries exactly ONE JSON line: native libraries (NCCL prints its version banner there) write to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    S.lib()  # fails loudly if the CUDA library is missing
    comm = None
    if world > 1:
        from tools.dist_helpers import broadcast_comm_id
        dist.init_process_group("nccl", device_id=dev)
        comm = S.Comm(broadcast_comm_id(S, rank, dev), world, rank, local)   # the data path's collectives are the library's own

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.cpu()]

    big = args.dataset == "synthetic"
    total = args.chains or TOTAL_CHAINS[args.dataset]
    burn = args.burn_calls or (1 if big else 5)
    samp = args.sample_calls or (1 if big else 5)
    algo = ALGO[args.dataset]
    job = Job(S, args.dataset, total, burn, samp, algo["k"], rank, world, local, comm)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def timed(job, run, steps, warmup, resident):
        """-> (wall s of `steps` steps, max over ranks; launches; sweep kernel ms per step; device ms per step)"""
        for _ in range(warmup):
            job.step_resident(run) if resident else job.step_e2e()
            flush.zero_()
        if run is not None:
            run.sync(); run.sweep_time(reset=True); run.elapsed_ms(reset=True)
            n0 = run.kernel_launches()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            job.step_resident(run) if resident else job.step_e2e()
            flush.zero_()                                              # L2 flush between timed iterations
        barrier()
        dt = time.perf_counter() - t0
        if run is None:
            return max_over_ranks([dt])[0], 0, 0.0, 0.0
        sweep_ms, n_sweep = run.sweep_time(reset=True)
        dev_ms = run.elapsed_ms(reset=True)
        launches = run.kernel_launches() - n0
        dt, sweep_ms, dev_ms = max_over_ranks([dt, sweep_ms / max(1, n_sweep), dev_ms / steps])
        return dt, launches, sweep_ms, dev_ms

    # ---- the headline workload
    run = job.make_run()
    clocks = ClockSampler(local)
    for _ in range(args.warmup):
        job.step_resident(run)
        flush.zero_()
    if rank == 0:
        clocks.start()
    dt, launches, sweep_ms, dev_ms = timed(job, run, args.steps, 0, True)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, job, run)
    run.close()
    dt_e2e, _, _, _ = timed(job, None, args.steps, args.warmup, False)

    # ---- `also`: config 5 as a full line at every N
    also = {}
    if not big and not args.no_synthetic:
        sj = Job(S, "synthetic", TOTAL_CHAINS["synthetic"], 1, 1, ALGO["synthetic"]["k"], rank, world, local, comm)
        srun = sj.make_run()
        s_dt, s_launches, s_sweep_ms, s_dev_ms = timed(sj, srun, 2, 1, True)
        srun.close()
        s_e2e, _, _, _ = timed(sj, None, 1, 1, False)
        if rank == 0:
            h2d, d2h = sj.bytes_per_step()
            sv = sj.sweeps_per_step * 2 / s_dt
            also["synthetic_65536"] = {
                "workload": workload_name("synthetic"), "value": sv, "unit": UNIT, "n_gpus": world, "scaling": "strong",
                "chains_total": sj.total, "chains_per_gpu": sj.n_local, "sweeps_per_chain_per_step": 20, "steps": 2, "warmup": 1,
                "ms_per_step": s_dt / 2 * 1e3, "gpu_launches": s_launches,
                "what": "init + (1 burn-in + 1 sampling call) x 10 sweeps + selection (k=2) + pair-order counts, large-shape kernel",
                "e2e": {"value": sj.sweeps_per_step / s_e2e, "unit": UNIT, "ms_per_step": s_e2e * 1e3, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "kernel": "ser_sweep_kernel_big", "kernel_ms_per_launch": s_sweep_ms,
                "kernel_sweeps_per_s_per_gpu": sj.n_local * 20 / (s_sweep_ms * 1e-3) if s_sweep_ms else None}

    if rank == 0:
        value = job.sweeps_per_step * args.steps / dt
        e2e_value = job.sweeps_per_step * args.steps / dt_e2e
        # roofline of the dominant kernel: CUDA events around every sweep launch of the timed region (one per step)
        mb = S.microbench(local)
        calls = burn + samp
        kernel_sweeps_per_s = job.n_local * calls * 10 / (sweep_ms * 1e-3)
        achieved = 10.0 * algo["F"] * kernel_sweeps_per_s / 1e12
        traffic = traffic_src = None
        if args.dataset in NCU_DRAM:
            nd = NCU_DRAM[args.dataset]
            if "per_item" in nd:   # one-thread-per-column kernel: work items x state round trip + the thinned samples
                slots = 148 * 3
                chunk = max(1, min(calls, job.n_local * calls // (32 * slots)))
                items = job.n_local * -(-calls // chunk)
                traffic = items * nd["per_item"] + job.n_local * samp * 2 * job.N
                traffic_src = ("%s: %.0f B of DRAM traffic per work item x %d items of one launch (%d calls per item) + %d thinned samples x %d B"
                               % (nd["src"], nd["per_item"], items, chunk, job.n_local * samp, 2 * job.N))
            else:
                traffic = nd["per_sweep"] * job.n_local * calls * 10
                traffic_src = "%s: %.0f B of DRAM traffic per chain-sweep x %d chain-sweeps of one launch" % (nd["src"], nd["per_sweep"], job.n_local * calls * 10)
        if "synthetic_65536" in also and also["synthetic_65536"]["kernel_sweeps_per_s_per_gpu"]:
            also["synthetic_65536"]["fp64_frac"] = 10.0 * ALGO["synthetic"]["F"] * also["synthetic_65536"]["kernel_sweeps_per_s_per_gpu"] / 1e12 / mb["fp64_tflops"]
        roofline = {
            "bound": "fp64", "achieved": achieved, "peak": mb["fp64_tflops"], "unit": "TFLOP/s",
            "frac": achieved / mb["fp64_tflops"], "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_per_launch": "10 F = %d fp64 flop per sweep (SURVEY 8d) x %d chain-sweeps" % (10 * algo["F"], job.n_local * calls * 10),
            "peak_source": "ser_microbench fp64 FMA on this GPU, measured live (MEASURED_PEAKS.json holds only HBM and bf16); "
                           "peak_kernels_ms are the kernel times the three SM-local peaks were derived from (work: include/seriation_b200.h)",
            "peak_kernels_ms": {"fp64": mb["fp64_kernel_ms"], "lds": mb["lds_kernel_ms"], "popc": mb["popc_kernel_ms"]},
            "kernel": "ser_sweep_kernel_big" if big else "ser_sweep_kernel", "kernel_ms_per_launch": sweep_ms, "launches_per_step": 1,
            "kernel_sweeps_per_s_per_gpu": kernel_sweeps_per_s, "device_ms_per_step_all_kernels": dev_ms,
            "smem": {"achieved_gbs": algo["B"] * kernel_sweeps_per_s / 1e9, "peak_gbs": mb["lds_gbs"],
                     "frac": algo["B"] * kernel_sweeps_per_s / 1e9 / mb["lds_gbs"]},
            "int_popc": {"achieved_gops": algo["C"] / 32 * kernel_sweeps_per_s / 1e9, "peak_gops": mb["popc_gops"],
                         "frac": algo["C"] / 32 * kernel_sweeps_per_s / 1e9 / mb["popc_gops"]},
            "hbm": {"achieved_gbs": algo["hbm_sample"] / 10 * kernel_sweeps_per_s / 1e9, "peak_gbs": _hbm_peak(),
                    "frac": algo["hbm_sample"] / 10 * kernel_sweeps_per_s / 1e9 / _hbm_peak()},
        }

    # ---- `also`: the reference's actual regime, one GPU: 1000 burn-in calls, then 1000 sampling calls, 1000 stored samples
    if world == 1 and not big and not args.no_stationary:
        also["stationary_1000+1000"] = stationary_regime(S, job, args.stationary_chains, local)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            procs = os.cpu_count() or 1
            ccalls = args.cpu_calls or auto_cpu_calls(args.dataset)
            v, kind = cpu_reference_run(args.dataset, ccalls, procs)
            cpu = {"value": v, "unit": UNIT, "cores": procs, "kind": kind, "sample": cpu_sample_text(procs, ccalls, args.dataset)}
        h2d, d2h = job.bytes_per_step()
        line = json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": ("synthetic 1024 x 4096 occurrence matrix (ser_dataset_synthetic), Philox free-running chains" if big else
                                     "NOW subset %s (committed fixture of the reference's Dataset/), Philox free-running chains" % args.dataset),
            "config": {"workload": workload_name(args.dataset), "arm": "B200: init + (%d burn-in + %d sampling) calls x 10 sweeps in one persistent launch "
                       "+ on-device selection (k=%d) + pair-order counts" % (burn, samp, algo["k"]),
                       "chains_total": total, "chains_per_gpu": job.n_local, "sweeps_per_step": job.sweeps_per_step,
                       "parallelism": "chains sharded x%d by global chain id; collectives: ncclAllGather of E[-logL] + ncclAllReduce of the PO counts, "
                                      "issued by the C library on the run's stream" % world if world > 1 else "one GPU",
                       "l2": "256 MB flush buffer written between timed steps"},
            "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                                   "ms_per_step": dt_e2e / args.steps * 1e3},
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "also": also or None,
        })
        sys.stdout.flush()
        os.write(json_fd, (line + "\n").encode())
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


def stationary_regime(S, job, n_chains, local):
    """the reference's own schedule (mcmc.c:107,140-143,180-185) on one GPU: 1000 burn-in calls from the randomised
    start, then 1000 sampling calls with all 1000 thinned samples stored, then the cross-chain step over T = 1000"""
    import numpy as np
    marks = []

    def mark(what):
        marks.append((what, time.perf_counter()))
    t0 = time.perf_counter()
    ds = S.Dataset.from_bits(job.X, job.hard)
    run = S.Run(ds, n_chains, mode=S.MODE_FREE, seed=20060206, store=S.STORE_PI, max_samples=1000, device=local)
    mark("create")
    run.init().advance(1000, False).sync()
    mark("burn-in")
    burn_ms, _ = run.sweep_time(reset=True)
    acc0 = np.sum([run.counters(i) for i in range(0, n_chains, max(1, n_chains // 64))], axis=0).astype(float)
    run.advance(1000, True).sync()
    mark("sampling")
    samp_ms, _ = run.sweep_time(reset=True)
    acc1 = np.sum([run.counters(i) for i in range(0, n_chains, max(1, n_chains // 64))], axis=0).astype(float)
    run.elapsed_ms(reset=True)
    res = run.cross_chain(job.k)
    mark("cross-chain")
    cc_ms = run.elapsed_ms(reset=True)
    d_ch = np.full(job.k, -1, np.int32); d_ch[:len(res["chosen"])] = res["chosen"]
    run.po_counts(d_ch)                                   # the pair-order kernel alone (+ its copies)
    import torch
    d_chosen = torch.from_numpy(d_ch).cuda(local)
    d_counts = torch.zeros((job.k, job.N, job.N), dtype=torch.int32, device="cuda:%d" % local)
    torch.cuda.synchronize()
    run.elapsed_ms(reset=True)
    run.po_counts_device(d_chosen.data_ptr(), job.k, d_counts.data_ptr())
    po_ms = run.elapsed_ms(reset=True)
    po = S.po_finalize(res["counts"][:max(1, len(res["chosen"]))], job.k) if len(res["chosen"]) else None
    ok = run.check() == 0
    run.close()
    mark("po probe + check + close")
    wall = time.perf_counter() - t0
    prev = t0
    for what, t in marks:
        print("stationary regime: %-26s %8.1f ms" % (what, (t - prev) * 1e3), file=sys.stderr)
        prev = t
    d = acc1 - acc0
    sw = max(d[7], 1.0)
    return {
        "workload": "%s, %d chains x (1000 burn-in + 1000 sampling calls x 10 sweeps), 1000 stored samples per chain, k=%d" % (job.dataset, n_chains, job.k),
        "burn_in_sweeps_per_s": n_chains * 10000 / (burn_ms * 1e-3), "stationary_sweeps_per_s": n_chains * 10000 / (samp_ms * 1e-3),
        "unit": UNIT, "sweep_kernel_ms": {"burn_in": burn_ms, "sampling": samp_ms},
        "e2e": {"value": n_chains * 20000 / wall, "unit": UNIT, "wall_s": wall,
                "what": "host dataset -> run creation -> init -> 20 000 sweeps per chain -> selection + pair-order counts over T = 1000 -> host"},
        "cross_chain_ms_T1000": cc_ms, "po_kernel_ms_T1000": po_ms, "sample_store_gb": n_chains * 1000 * job.N * 2 / 1e9,
        "acceptance_in_sampling_phase": {"ab_changed_per_taxon_step": d[2] / (sw * 2 * job.M), "pi1": d[3] / (sw * 5), "pi2": d[4] / (sw * 5),
                                         "swap": d[5] / sw, "pi3": d[6] / (sw * 5)},
        "consistent": ok, "po_diag_ok": bool(po is not None and (np.diag(po) < 0).all()),
    }


def _hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0  # fallback stated in B200_PROFILING.md


if __name__ == "__main__":
    main()
