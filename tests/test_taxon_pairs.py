"""Taxon pair relations on the device (ser_run_taxon_pairs, one-shot and streaming through ser_run_accumulate with SER_ACC_TAXA):
first / last appearance order, superposition and coexistence of every pair of taxa, checked against numpy over the stored samples and
over crafted stores injected through a checkpoint, with the exact identities of the contract."""
import ctypes as C
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, load_hex_dataset, random_dataset
from test_checkpoint import _layout, _patch_record
from test_reductions import _crafted_ab

E_ARG, E_STATE = -1, -4
KEYS = ("first", "last", "precedes", "coexist")


@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


def _raises(S, code, fn, *args, **kw):
    with pytest.raises(S.SeriationError) as e:
        fn(*args, **kw)
    assert str(e.value).startswith("[%d]" % code), str(e.value)
    return str(e.value)


def _ptr(a, t=C.c_int32):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


# ----------------------------------------------------------------------------- numpy reference and identities
def _ref_taxon_pairs(a, b):
    """the four [M][M] counts over rows t of a, b [T][M]: broadcast comparisons summed over t (one row at a time)"""
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    M = a.shape[1]
    out = {key: np.zeros((M, M), np.int64) for key in KEYS}
    for t in range(a.shape[0]):
        am, an, bm, bn = a[t][:, None], a[t][None, :], b[t][:, None], b[t][None, :]
        out["first"] += am < an
        out["last"] += bm < bn
        out["precedes"] += bm <= an
        out["coexist"] += np.maximum(am, an) < np.minimum(bm, bn)
    return out


def _check_identities(tp, a, b):
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    T, M = a.shape
    eq_a = sum((a[t][:, None] == a[t][None, :]).astype(np.int64) for t in range(T)) if T else np.zeros((M, M), np.int64)
    eq_b = sum((b[t][:, None] == b[t][None, :]).astype(np.int64) for t in range(T)) if T else np.zeros((M, M), np.int64)
    first, last, prec, co = (np.asarray(tp[key], np.int64) for key in KEYS)
    assert np.array_equal(first + first.T + eq_a, np.full((M, M), T))
    assert np.array_equal(last + last.T + eq_b, np.full((M, M), T))
    assert np.array_equal(co, co.T)
    assert not np.diag(first).any() and not np.diag(last).any()
    assert np.array_equal(np.diag(prec), (a == b).sum(axis=0)) and np.array_equal(np.diag(co), (a < b).sum(axis=0))
    full = (a < b).all(axis=0)                              # taxa whose range is never empty
    both = full[:, None] & full[None, :]
    assert np.array_equal((co + prec + prec.T)[both], np.full(both.sum(), T))


# ----------------------------------------------------------------------------- CPU
def test_reference_on_hand_written_cases():
    # N = 5: [1, 3) and [3, 5) touch at 3 (precedes, not coexist); [2, 2) is empty; [0, 5) holds [1, 3)
    a, b = np.array([[1, 3, 2, 0]]), np.array([[3, 5, 2, 5]])
    r = _ref_taxon_pairs(a, b)
    assert r["first"].tolist() == [[0, 1, 1, 0], [0, 0, 0, 0], [0, 1, 0, 0], [1, 1, 1, 0]]
    assert r["last"].tolist() == [[0, 1, 0, 1], [0, 0, 0, 0], [1, 1, 0, 1], [0, 0, 0, 0]]
    assert r["precedes"].tolist() == [[0, 1, 0, 0], [0, 0, 0, 0], [0, 1, 1, 0], [0, 0, 0, 0]]
    assert r["coexist"].tolist() == [[1, 0, 0, 1], [0, 1, 0, 1], [0, 0, 0, 0], [1, 1, 0, 1]]
    _check_identities(r, a, b)
    # empty ranges at 0 and at N = 5, and the whole range
    a, b = np.array([[0, 5, 0]]), np.array([[0, 5, 5]])
    r = _ref_taxon_pairs(a, b)
    assert r["first"].tolist() == [[0, 1, 0], [0, 0, 0], [0, 1, 0]]
    assert r["last"].tolist() == [[0, 1, 1], [0, 0, 0], [0, 0, 0]]
    assert r["precedes"].tolist() == [[1, 1, 1], [0, 1, 0], [0, 1, 0]]
    assert r["coexist"].tolist() == [[0, 0, 0], [0, 0, 0], [0, 0, 1]]
    _check_identities(r, a, b)
    # two samples: disjoint ranges, then equal ones (ties in a and in b)
    a, b = np.array([[0, 4], [1, 1]]), np.array([[2, 6], [4, 4]])
    r = _ref_taxon_pairs(a, b)
    assert r["first"].tolist() == r["last"].tolist() == r["precedes"].tolist() == [[0, 1], [0, 0]]
    assert r["coexist"].tolist() == [[2, 1], [1, 2]]
    _check_identities(r, a, b)


def test_reference_identities_on_random_ranges():
    rng = np.random.default_rng(3)
    for N, M, T in ((2, 1, 1), (5, 7, 40), (12, 33, 17)):
        lo, hi = np.sort(rng.integers(0, N + 1, (2, T, M)), axis=0)
        _check_identities(_ref_taxon_pairs(lo, hi), lo, hi)
        hi = np.maximum(hi, lo + 1)                                  # no empty range: the three-way identity holds everywhere
        ok = hi <= N
        lo, hi = np.where(ok, lo, N - 1), np.where(ok, hi, N)
        r = _ref_taxon_pairs(lo, hi)
        assert np.array_equal(r["coexist"] + r["precedes"] + r["precedes"].T, np.full((M, M), T))


def test_argument_checks_without_a_device(S):
    L = S.lib()
    chosen, out, n = np.zeros(1, np.int32), np.zeros(64, np.int32), np.zeros(1, np.int32)
    assert L.ser_run_taxon_pairs(None, _ptr(chosen), 1, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_accumulate(None, 128) == E_ARG


def test_taxon_pair_kernel_is_built_for_sm100a_without_stack_or_spills(S):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump is not installed")
    out = subprocess.run([exe, "-res-usage", S.LIB_PATH], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    lines = out.splitlines()
    idx = [i for i, ln in enumerate(lines) if "Function" in ln and "ser_taxon_pair_kernel" in ln]
    assert len(idx) == 1
    res = lines[idx[0] + 1]
    assert "STACK:0" in res and "LOCAL:0" in res, res


def test_cli_taxon_pairs_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--taxon-pairs", str(tmp_path / "t")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "usage" in r.stderr and not (tmp_path / "t.first.csv").exists()


# ----------------------------------------------------------------------------- GPU
def _check_run(run, chosen, local=None):
    """taxon_pairs of `chosen` against the reference over each chain's fetched samples, and the identities"""
    tp = run.taxon_pairs(chosen)
    for c, g in enumerate(chosen):
        s = run.fetch_samples(g if local is None else local[c])
        assert tp["n_samples"][c] == s["a"].shape[0], g
        want = _ref_taxon_pairs(s["a"], s["b"])
        for key in KEYS:
            assert np.array_equal(tp[key][c], want[key]), (g, key)
        _check_identities({key: tp[key][c] for key in KEYS}, s["a"], s["b"])
    return tp


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["g10s10", "g2s2", "big", "synthetic", "manycd"])
def test_one_shot_equals_numpy(S, case, monkeypatch):
    if case == "big":
        monkeypatch.setenv("SER_FORCE_BIG", "256")
    if case == "synthetic":
        ds, n, burn, T, spc, chosen = S.Dataset.synthetic(1024, 4096, 16), 3, 2, 4, 1, [2, 0]
    else:
        name = "g2s2" if case == "g2s2" else "g10s10"
        ds, n, burn, T, spc, chosen = S.Dataset.from_bits(*load_hex_dataset(name)), 6, 20, 77, 10, [4, 1, 5]
    run = S.Run(ds, n, seed=11, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T, manycd=case == "manycd")
    run.init().advance(burn, False).advance(T, True).sync()
    assert (run.kernel_path() == 0) == (case not in ("big", "synthetic"))
    _check_run(run, chosen)


@pytest.mark.gpu
def test_one_shot_on_the_reference_tape(S):
    g = np.load(os.path.join(GOLDEN, "ref_g10s10.npz"))
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    calls = len(g["kind"]) - 1
    run = S.Run(ds, 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls).set_tapes([g["tape"]]).init().advance(calls, True).sync()
    tp = _check_run(run, [0])
    assert tp["n_samples"][0] == calls


@pytest.mark.gpu
@pytest.mark.parametrize("M", [1, 31, 32, 33, 95])
def test_crafted_stores_through_a_checkpoint(S, tmp_path, M):
    """tile edges in M, staging edges in T (each chain its own T), empty ranges and the (0, N), (N, N) pairs"""
    N, n, R = 40, 5, 65
    X, hard = random_dataset(np.random.default_rng(M), N, M, 3, .15)
    ds = S.Dataset.from_bits(X, hard)
    kw = dict(seed=5, store=S.STORE_FULL, max_samples=R)
    f = str(tmp_path / "ck")
    S.Run(ds, n, **kw).init().advance(2, False).advance(R, True).save_checkpoint(f).close()
    data = open(f, "rb").read()
    assert _layout(N, M, 0, S.STORE_FULL, R, 0)["size"] == struct.unpack_from("<Q", data, 88)[0]
    rng = np.random.default_rng(N * M)
    own = [1, 31, 32, 33, 65]
    crafted = {}
    for c in range(n):
        a, b = _crafted_ab(rng, N, M, R)
        crafted[c] = (a[:own[c]], b[:own[c]])

        def edit(rec, L, a=a, b=b, t=own[c]):
            rec[L["sa"]:L["sa"] + a.nbytes] = a.tobytes()
            rec[L["sb"]:L["sb"] + b.nbytes] = b.tobytes()
            struct.pack_into("<i", rec, 156, t)
        patched = _patch_record(f, c, edit)
        open(f, "wb").write(patched)
    run = S.Run(ds, n, **kw).load_checkpoint(f)
    chosen = [4, 2, 0, 3, 1]
    tp = run.taxon_pairs(chosen)
    assert tp["n_samples"].tolist() == [own[g] for g in chosen]
    for c, g in enumerate(chosen):
        a, b = crafted[g]
        want = _ref_taxon_pairs(a, b)
        for key in KEYS:
            assert np.array_equal(tp[key][c], want[key]), (M, g, key)
        _check_identities({key: tp[key][c] for key in KEYS}, a, b)
    assert run.check() == 0


@pytest.mark.gpu
def test_slab_convention_and_subsets(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    M = ds.M
    run = S.Run(ds, 0, seed=2, store=S.STORE_FULL, max_samples=20, chain_ids=[7, 30]).init().advance(3, False).advance(20, True).sync()
    want = run.taxon_pairs([7, 30])
    chosen = np.array([30, -1, 8, 7], np.int32)
    k = len(chosen)
    outs = [np.full((k, M, M), 7, np.int32) for _ in KEYS]
    n = np.full(k, 7, np.int32)
    assert S.lib().ser_run_taxon_pairs(run._h, _ptr(chosen), k, *(_ptr(o) for o in outs), _ptr(n)) == 0
    assert n.tolist() == [20, 0, 0, 20]
    for o, key in zip(outs, KEYS):
        assert np.all(o[1] == 7) and np.all(o[2] == 7), key
        assert np.array_equal(o[0], want[key][1]) and np.array_equal(o[3], want[key][0]), key
    # every subset of the outputs: the requested ones as above, the others unwritten
    for mask in range(1, 16):
        ask = [bool(mask >> q & 1) for q in range(4)]
        outs = [np.full((1, M, M), 7, np.int32) if w else None for w in ask]
        n1 = np.zeros(1, np.int32)
        assert S.lib().ser_run_taxon_pairs(run._h, _ptr(np.array([30], np.int32)), 1, *(_ptr(o) for o in outs), _ptr(n1)) == 0
        assert n1[0] == 20
        for o, key in zip(outs, KEYS):
            if o is not None:
                assert np.array_equal(o[0], want[key][1]), (mask, key)
        got = run.taxon_pairs([30], **dict(zip(KEYS, ask)))
        assert [got[key] is None for key in KEYS] == [not w for w in ask]


def _same(x, y, what):
    for key in KEYS + ("n_samples",):
        assert np.array_equal(x[key], y[key]), (what, key)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["g10s10", "33x70"])
def test_streaming_equals_one_shot(S, shape):
    if shape == "g10s10":
        ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    else:
        ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(70), 33, 70, 3, .12))
    burn, T, chosen = 5, 70, [1, 4, 99]                     # 99: held by no run here
    ref = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    want = ref.taxon_pairs(chosen)
    assert want["n_samples"].tolist() == [T, T, 0]
    for W in (1, 7, 64):
        whole = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=W).init().accumulate(po=False, sums=False, taxon_pairs=True)
        whole.advance(burn, False).advance(T, True).sync()
        _same(whole.taxon_pairs(chosen), want, ("contiguous", W))
        sub = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=W, chain_ids=[4, 1]).init().accumulate(taxon_pairs=True, ranges=True)
        sub.advance_both(burn, 5).advance(T - 5, True).sync()  # 5 and 65 samples: neither a multiple of 7 or 64
        _same(sub.taxon_pairs(chosen), want, ("subset", W))
        whole.close()
        sub.close()
    odd = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=16, chain_ids=[1, 4]).init().accumulate(po=False, sums=False, taxon_pairs=True)
    odd.advance_both(burn, 7).advance(20, True).advance(43, True).sync()
    _same(odd.taxon_pairs(chosen), want, "advances off the window")


@pytest.mark.gpu
def test_replay_chosen_and_pooled_probabilities(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, samp, k = 64, 20, 30, 3
    one = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_FULL)
    chosen = S.choose_chains(one, k)
    want = one.run.taxon_pairs(chosen)
    first = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_NONE)
    two = S.replay_chosen(first, chosen, window=16, taxon_pairs=True)
    assert two.run.cfg.store == S.STORE_FULL
    _same(two.run.taxon_pairs(chosen), want, "replay_chosen")
    x, y = S.taxon_pairs(two, chosen), S.taxon_pairs(one, chosen)
    assert x["n_samples"] == y["n_samples"] == k * samp
    for key in KEYS:
        pooled = want[key].sum(axis=0, dtype=np.int64)
        assert np.array_equal(x["counts"][key], pooled) and np.array_equal(y["counts"][key], pooled), key
        assert np.array_equal(x[key], pooled / (k * samp)) and np.array_equal(x[key], y[key]), key
        assert x[key].dtype == np.float64 and np.all((x[key] >= 0) & (x[key] <= 1)), key


@pytest.mark.gpu
def test_checkpoint_mid_window(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    burn, T, W, chosen = 5, 50, 16, [0, 2]
    flags = dict(po=True, sums=False, ranges=True, taxon_pairs=True)
    kw = dict(seed=8, store=S.STORE_FULL, max_samples=W)
    whole = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(T, True).sync()
    want = whole.taxon_pairs(chosen)
    whole.save_checkpoint(str(tmp_path / "whole.ckpt"))
    part = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(23, True)
    part.save_checkpoint(str(tmp_path / "part.ckpt"))
    rest = S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint(str(tmp_path / "part.ckpt")).advance(T - 23, True).sync()
    _same(rest.taxon_pairs(chosen), want, "resumed")
    rest.save_checkpoint(str(tmp_path / "rest.ckpt"))
    assert (tmp_path / "rest.ckpt").read_bytes() == (tmp_path / "whole.ckpt").read_bytes()
    # a run accumulating other flags does not load it, and neither does one that adds the flag to a file without it
    other = S.Run(ds, 3, **kw).accumulate(po=True, sums=False, ranges=True)
    _raises(S, E_STATE, other.load_checkpoint, str(tmp_path / "part.ckpt"))
    plain = S.Run(ds, 3, **kw).init().accumulate(po=True, sums=False, ranges=True).advance(burn, False).advance(9, True)
    plain.save_checkpoint(str(tmp_path / "plain.ckpt"))
    _raises(S, E_STATE, S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint, str(tmp_path / "plain.ckpt"))


@pytest.mark.gpu
def test_checkpoint_record_above_the_staging_size(S, tmp_path):
    """at 1024 x 4096 the taxon pair part alone is 256 MiB, so one record is larger than the 256 MiB a save or load stages through"""
    ds = S.Dataset.synthetic(1024, 4096, 16)
    kw = dict(seed=9, sweeps_per_call=1, store=S.STORE_FULL, max_samples=4, chain_ids=[5])
    flags = dict(po=False, sums=False, taxon_pairs=True)
    whole = S.Run(ds, 0, **kw).init().accumulate(**flags).advance(1, False).advance(9, True).sync()
    want = whole.taxon_pairs([5])
    whole.close()
    f = str(tmp_path / "big.ckpt")
    S.Run(ds, 0, **kw).init().accumulate(**flags).advance(1, False).advance(6, True).save_checkpoint(f).close()
    size = struct.unpack_from("<Q", open(f, "rb").read(104), 88)[0]
    assert size > 256 << 20
    rest = S.Run(ds, 0, **kw).accumulate(**flags).load_checkpoint(f).advance(3, True).sync()
    _same(rest.taxon_pairs([5]), want, "resumed large record")
    assert want["n_samples"].tolist() == [9]


@pytest.mark.gpu
def test_same_batch_twice_gives_the_same_bytes(S):
    ds = S.Dataset.synthetic(256, 700, 8)
    outs = []
    for _ in range(2):
        run = S.Run(ds, 3, seed=21, sweeps_per_call=2, store=S.STORE_FULL, max_samples=40).init().advance(3, False).advance(40, True).sync()
        outs.append(run.taxon_pairs([2, 0, 1]))
        outs.append(run.taxon_pairs([2, 0, 1]))
        run.close()
    for o in outs[1:]:
        for key in KEYS:
            assert o[key].tobytes() == outs[0][key].tobytes(), key


@pytest.mark.gpu
def test_refusals_launch_nothing(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=8).init().advance(8, True).sync()
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate(ranges=True).advance(8, True).sync()
    fresh = S.Run(ds, 2, store=S.STORE_FULL, max_samples=8)
    for run, msg in ((pi_only, "SER_STORE_FULL"), (acc, "SER_ACC_TAXA"), (fresh, "not initialised")):
        before = run.kernel_launches()
        assert msg in _raises(S, E_STATE, run.taxon_pairs, [0])
        assert run.kernel_launches() == before, msg
    assert "SER_STORE_FULL" in _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_PI, max_samples=4).init().accumulate, taxon_pairs=True)
    run = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init()
    before = run.kernel_launches()
    L = S.lib()
    chosen, out, n = np.zeros(1, np.int32), np.zeros((1, ds.M, ds.M), np.int32), np.zeros(1, np.int32)
    assert L.ser_run_taxon_pairs(run._h, _ptr(chosen), 1, None, None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_taxon_pairs(run._h, _ptr(chosen), 0, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_taxon_pairs(run._h, None, 1, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_taxon_pairs(run._h, _ptr(chosen), 1, None, None, None, _ptr(out), None) == E_ARG
    for bad in (64, 256, 128 | 64):                      # SER_ACC_TAXA is bit 128; 64 and the bits above 128 are not flags
        assert L.ser_run_accumulate(run._h, bad) == E_ARG, bad
    assert run.kernel_launches() == before


@pytest.mark.gpu
def test_multi_device_slabs_sum_to_one_device(S):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, T, chosen = 64, 10, 25, [3, 40, 63]
    one = S.Run(ds, n, seed=6, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    want = one.taxon_pairs(chosen)
    m = S.Multi(ds, n, 2, seed=6, store=S.STORE_FULL, max_samples=T).init().advance(burn, T).sync()
    runs = {}
    for g in chosen:
        r, _ = m.locate(g)
        runs[r._h.value] = r
    assert len(runs) == 2
    parts = [r.taxon_pairs(chosen) for r in runs.values()]
    _same({key: sum(p[key] for p in parts) for key in KEYS + ("n_samples",)}, want, "ser_multi over 2 GPUs")


@pytest.mark.gpu
def test_cli_taxon_pairs(S, tmp_path):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp, M = 20, 60, X.shape[1]
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "2",
            "--dataset", str(tmp_path / "g10s10.txt"), "--window", "16"]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env, cwd=tmp_path).stdout.splitlines()
    pick = lambda lines, head: [x for x in lines if x.startswith(head)]
    out = run(["--taxon-pairs", str(tmp_path / "T")])
    line = pick(out, "taxon pairs:")
    assert len(line) == 1 and "coexist with P >= 0.95" in line[0]
    batch = S.run_all_chains(S.Dataset.from_bits(X, hard), 64, burn, samp, seed=0, store=S.STORE_FULL)
    chosen = S.choose_chains(batch, 2)
    assert ("chosen " + " ".join(map(str, chosen))) in pick(out, "selection:")[0]
    tp = S.taxon_pairs(batch, chosen)
    for key in KEYS:
        want = "".join(",".join("%.6f" % v for v in row) + "\n" for row in tp[key])
        assert (tmp_path / ("T.%s.csv" % key)).read_text() == want, key
    assert len(tp["first"]) == M
    co = tp["coexist"][np.triu_indices(M, 1)]
    assert "%d coexist with P >= 0.95 and %d with P <= 0.05" % ((co >= 0.95).sum(), (co <= 0.05).sum()) in line[0]
    # one replay serves both flags: the marginal files and po.csv do not change
    run(["--replay-selected", "--po", str(tmp_path / "p1.csv"), "--marginals", str(tmp_path / "P")])
    out2 = run(["--replay-selected", "--po", str(tmp_path / "p2.csv"), "--marginals", str(tmp_path / "Q"), "--taxon-pairs", str(tmp_path / "U")])
    assert (tmp_path / "p2.csv").read_bytes() == (tmp_path / "p1.csv").read_bytes()
    for suffix in (".sites.csv", ".taxa.csv"):
        assert (tmp_path / ("Q" + suffix)).read_bytes() == (tmp_path / ("P" + suffix)).read_bytes()
    for key in KEYS:
        assert (tmp_path / ("U.%s.csv" % key)).read_bytes() == (tmp_path / ("T.%s.csv" % key)).read_bytes()
    assert pick(out2, "taxon pairs:") == line
