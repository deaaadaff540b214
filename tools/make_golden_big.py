#!/usr/bin/env python
"""tests/golden/ref_synthetic_1024x4096.npz: BASELINE.json config 5's shape against the UNMODIFIED reference.

Run in the build container (needs /root/reference and oracle/_ref/ref_mcmc_big = the reference's own mcmc.c
compiled with MAXS raised so that it can read 8 192-character rows, oracle/Makefile):
    python tools/make_golden_big.py

For 8 seeds the reference runs 10 mcmc_sample() calls (100 sweeps) on the deterministic 1024 x 4096 synthetic
matrix (ser_dataset_synthetic, seed 0x5EB1A710, 16 hard sites) under the recording GSL shim; the full model
state after the randomised start and after every call is committed (a, b and pi in full for the first seed, as CRC32s
for all eight).  The draw tapes themselves (53 MB) are not:
the shim's MT19937 is reproduced by the oracle's own MT source, so a test regenerates the tape from the seed,
checks its length and checksum against the values stored here, and replays it on the GPU."""
import os
import sys
import tempfile
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import seriation_b200 as S  # noqa: E402  (host-only entry points: the synthetic generator)
from oracle import oracle as O  # noqa: E402
from tools.datasets import write_txt  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "ref_synthetic_1024x4096.npz")
SEEDS = list(range(101, 109))
CALLS = 10


def one(args):
    seed, path = args
    with tempfile.TemporaryDirectory() as td:
        dims, states, tape = O.ref_trace(path, 0, CALLS, td, seed=seed, binary=O.REF_BIN + "_big")
    return seed, states, tape


if __name__ == "__main__":
    O.build()
    X, hard = S.Dataset.synthetic(1024, 4096, 16).arrays()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "synthetic.txt")
        write_txt(path, X, hard)
        with ThreadPoolExecutor(8) as ex:
            res = list(ex.map(one, [(s, path) for s in SEEDS]))
    out = {}
    for k in ("a", "b", "pi"):   # every chain's states as CRC32s of their int16 bytes, the first chain's in full (file < 1 MB)
        v = np.stack([np.stack([getattr(st, k) for st in states]) for _, states, _ in res]).astype(np.int16)
        out[k], out[k + "_crc"] = v[:1], np.array([[zlib.crc32(rec.tobytes()) for rec in chain] for chain in v], np.int64)
    out["tot"] = np.stack([np.stack([st.tot for st in states]) for _, states, _ in res]).astype(np.int32)
    out["cdl"] = np.array([[[st.c, st.d, st.loglik] for st in states] for _, states, _ in res])
    out["slots"] = np.array([[st.slots for st in states] for _, states, _ in res], np.int64)
    out["tape_len"] = np.array([t.size for _, _, t in res], np.int64)
    out["tape_crc"] = np.array([zlib.crc32(t.tobytes()) for _, _, t in res], np.int64)
    out["seeds"] = np.array(SEEDS, np.int64)
    out["x_crc"] = np.array([zlib.crc32(X.tobytes()), zlib.crc32(hard.tobytes())], np.int64)
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, os.path.getsize(OUT), "bytes; records per chain", out["a"].shape[1], "tape slots", out["tape_len"].tolist())
