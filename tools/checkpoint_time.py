"""Cost of a checkpoint on one GPU: wall time of ser_run_save_checkpoint and ser_run_load_checkpoint, and the file size, for
runs without a sample store (the live state alone).

    python tools/checkpoint_time.py [--dir DIR] [--out FILE.json] [--quick]

Cases: 16 384 chains of g2s2, and 65 536 chains of the 1024 x 4096 synthetic matrix (BASELINE.json config 5).  Each run is
initialised and advanced one call, then saved (host clock around the call, which waits for the run's stream, writes path.tmp,
fsyncs it and renames it), then loaded into a fresh run (host clock around the call, which ends with the consistency check
and a synchronise).  The loaded run is saved again and the two files must be byte-identical.  The files go to --dir (default:
a temporary directory); the times include that file system.  --quick shrinks the cases to a rehearsal.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import seriation_b200 as S  # noqa: E402
from tools.datasets import load_hex_dataset  # noqa: E402


def case(label, ds, n, d, reps):
    path, again = os.path.join(d, "ck"), os.path.join(d, "ck2")
    run = S.Run(ds, n, seed=20060206).init().advance(1, False).sync()
    save = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run.save_checkpoint(path)
        save.append(time.perf_counter() - t0)
    run.close()
    load = []
    for _ in range(reps):
        fresh = S.Run(ds, n, seed=20060206)
        t0 = time.perf_counter()
        fresh.load_checkpoint(path)
        load.append(time.perf_counter() - t0)
        fresh.save_checkpoint(again)
        fresh.close()
        with open(path, "rb") as a, open(again, "rb") as b:
            assert a.read() == b.read(), "a loaded run saves a different file"
    size = os.path.getsize(path)
    row = dict(case=label, N=ds.N, M=ds.M, chains=n, file_bytes=size, bytes_per_chain=size / n, save_s=save, load_s=load)
    print(json.dumps(row), flush=True)
    os.remove(path)
    os.remove(again)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--dir", help="where the checkpoint files are written (default: a temporary directory)")
    ap.add_argument("--out", help="also write the results as JSON here")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("checkpoint_time: needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    res = dict(gpu=gpu, cases=[])
    with tempfile.TemporaryDirectory(dir=a.dir) as d:
        res["cases"].append(case("g2s2", S.Dataset.from_bits(*load_hex_dataset("g2s2")), 256 if a.quick else 16384, d, a.reps))
        res["cases"].append(case("synthetic 1024x4096 (config 5)", S.Dataset.synthetic(1024, 4096, 16), 256 if a.quick else 65536, d, a.reps))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print("gpu:", gpu)


if __name__ == "__main__":
    main()
