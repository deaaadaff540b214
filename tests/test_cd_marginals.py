"""Posterior of the error rates c, d on the device (ser_run_cd_marginals, one-shot and streaming through ser_run_accumulate with
SER_ACC_CD): per taxon on a manycd run, the scalar pair otherwise, the exp sums and the log-scale histograms checked against numpy over
the stored samples, over the reference's recorded trace and over crafted stores injected through a checkpoint, and the exact identity
with ser_run_chain_stats' e_c and e_d."""
import ctypes as C
import os
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_hex_dataset, random_dataset
from test_checkpoint import _patch_record

E_ARG, E_STATE = -1, -4
KEYS = ("c_sum", "d_sum", "c_hist", "d_hist")
BOUNDS = dict(c=(-6.9077552789821368, -2.3025850929940455), d=(-1.6094379124341003, -0.22314355131420971))
B = 256


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


# ----------------------------------------------------------------------------- numpy reference of the contract
def _bins(x, name):
    """bin = min(B - 1, floor((x - lo) * s)), s = B / (hi - lo), each step rounded to nearest; x <= lo and NaN -> 0"""
    lo, hi = BOUNDS[name]
    s = B / (hi - lo)
    with np.errstate(invalid="ignore"):
        y = (np.asarray(x, np.float64) - lo) * s
        y = np.where(y > 0, y, 0.0)
    return np.minimum(np.floor(y), B - 1).astype(np.int64)


def _ref(c, d):
    """sums (sequential fold of exp in sample order from 0.0) and histograms [R][B] over rows t of c, d [T][R]"""
    out = {}
    for name, x in (("c", np.asarray(c, np.float64)), ("d", np.asarray(d, np.float64))):
        T, R = x.shape
        s = np.zeros(R)
        with np.errstate(over="ignore", invalid="ignore"):
            for t in range(T):
                s = s + np.exp(x[t])
        j = _bins(x, name)
        h = np.zeros((R, B), np.int64)
        for r in range(R):
            h[r] = np.bincount(j[:, r], minlength=B)
        out[name + "_sum"], out[name + "_hist"] = s, h
    return out


def _compare(got, want, c, what):
    """exact counts, sums within 1e-13 relative (numpy's exp is not the device's), every row summing to T"""
    T = want["c_hist"].sum(axis=1)[0] if len(want["c_hist"]) else 0
    for name in ("c", "d"):
        assert np.array_equal(got[name + "_hist"][c], want[name + "_hist"]), (what, name)
        assert np.all(got[name + "_hist"][c].sum(axis=1) == T), (what, name)
        np.testing.assert_allclose(got[name + "_sum"][c], want[name + "_sum"], rtol=1e-13, atol=0, equal_nan=True, err_msg=str((what, name)))


# ----------------------------------------------------------------------------- CPU
def _interior_edge(name, j):
    """the smallest double whose bin is j (j > 0) under the contract's arithmetic, and the double below it"""
    lo, hi = BOUNDS[name]
    x = lo + j * (hi - lo) / B
    while _bins([x], name)[0] >= j:
        x = np.nextafter(x, -np.inf)
    while _bins([x], name)[0] < j:
        x = np.nextafter(x, np.inf)
    return x, np.nextafter(x, -np.inf)


def test_reference_on_hand_written_values():
    for name in ("c", "d"):
        lo, hi = BOUNDS[name]
        edge, below_edge = _interior_edge(name, 128)
        x = [lo, hi, np.nextafter(hi, -np.inf), edge, below_edge, lo - 0.5, np.nextafter(lo, -np.inf), hi + 0.5, np.nan, -np.inf,
             np.nextafter(lo, np.inf)]
        assert _bins(x, name).tolist() == [0, B - 1, B - 1, 128, 127, 0, 0, B - 1, 0, 0, 0], name
        s = B / (hi - lo)
        assert (edge - lo) * s >= 128 > (below_edge - lo) * s
        r = _ref(np.array(x)[:, None], np.array(x)[:, None])
        assert r[name + "_hist"].sum() == len(x) and r[name + "_hist"][0, 128] == 1 and r[name + "_hist"][0, 127] == 1
        assert r[name + "_hist"][0, 0] == 6 and r[name + "_hist"][0, B - 1] == 3
    # every row sums to T; the sum is the fold in sample order
    rng = np.random.default_rng(1)
    c = rng.uniform(*BOUNDS["c"], (37, 5))
    d = rng.uniform(*BOUNDS["d"], (37, 5))
    r = _ref(c, d)
    assert np.all(r["c_hist"].sum(axis=1) == 37) and np.all(r["d_hist"].sum(axis=1) == 37)
    fold = 0.0
    for t in range(37):
        fold = fold + np.exp(c[t, 3])
    assert r["c_sum"][3] == fold


def test_header_bounds_equal_the_python_constants():
    import seriation_b200 as S
    text = open(os.path.join(ROOT, "include", "seriation_b200.h")).read()
    got = {k: v for k, v in re.findall(r"#define (SER_M(?:IN|AX)[CD]) \(([-0-9.eE]+)\)", text)}
    assert {k: float(v) for k, v in got.items()} == dict(SER_MINC=S.MINC, SER_MAXC=S.MAXC, SER_MIND=S.MIND, SER_MAXD=S.MAXD)
    assert (S.MINC, S.MAXC) == BOUNDS["c"] and (S.MIND, S.MAXD) == BOUNDS["d"] and S.CD_BOUNDS == BOUNDS
    assert int(re.search(r"#define SER_CD_BINS (\d+)", text).group(1)) == S.CD_BINS == B
    assert int(re.search(r"#define SER_ACC_CD (\d+)", text).group(1)) == S.ACC_CD == 512
    assert np.allclose(np.exp([S.MINC, S.MAXC, S.MIND, S.MAXD]), [.001, .1, .2, .8], rtol=1e-15)
    assert S.cd_bin_edges("c")[0] == S.MINC and abs(S.cd_bin_edges("c")[-1] - S.MAXC) < 1e-15


def test_argument_checks_without_a_device(S):
    L = S.lib()
    chosen, s, n = np.zeros(1, np.int32), np.zeros(1), np.zeros(1, np.int32)
    assert L.ser_run_cd_marginals(None, _ptr(chosen), 1, _ptr(s, C.c_double), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_accumulate(None, 512) == E_ARG


def test_cd_hist_kernel_is_built_for_sm100a_without_stack_or_spills(S):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump is not installed")
    out = subprocess.run([exe, "-res-usage", S.LIB_PATH], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    lines = out.splitlines()
    idx = [i for i, ln in enumerate(lines) if "Function" in ln and "ser_cd_hist_kernel" in ln]
    assert len(idx) == 1
    res = lines[idx[0] + 1]
    assert "STACK:0" in res and "LOCAL:0" in res, res


def test_cli_cd_marginals_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--cd-marginals", str(tmp_path / "cd.csv")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "usage" in r.stderr and not (tmp_path / "cd.csv").exists()


# ----------------------------------------------------------------------------- GPU
def _stored(run, chain):
    """the stored c, d rows [T][R] of a local chain: per taxon on a manycd run, the scalar pair otherwise"""
    s = run.fetch_samples(chain)
    if run.manycd:
        return s["c_all"], s["d_all"]
    return s["c"][:, None], s["d"][:, None]


def _check_run(run, chosen, local=None):
    got = run.cd_marginals(chosen)
    for c, g in enumerate(chosen):
        cs, ds = _stored(run, g if local is None else local[c])
        assert got["n_samples"][c] == len(cs), g
        _compare(got, _ref(cs, ds), c, g)
    return got


def _check_identity(run, got, chosen):
    """on a run whose samples all fit the store: c_sum[:, 0] / T == e_c and d_sum[:, 0] / T == e_d, bit for bit"""
    st = run.chain_stats()
    for c, g in enumerate(chosen):
        T = float(got["n_samples"][c])
        assert (got["c_sum"][c, 0] / T).tobytes() == st["e_c"][g].tobytes(), g
        assert (got["d_sum"][c, 0] / T).tobytes() == st["e_d"][g].tobytes(), g


@pytest.mark.gpu
@pytest.mark.parametrize("case,manycd", [("g10s10", False), ("g10s10", True), ("g2s2", True), ("big", False), ("big", True),
                                         ("synthetic", True)])
def test_one_shot_equals_numpy(S, case, manycd, monkeypatch):
    if case == "big":
        monkeypatch.setenv("SER_FORCE_BIG", "256")
    if case == "synthetic":
        ds, n, burn, T, spc, chosen = S.Dataset.synthetic(1024, 4096, 16), 3, 2, 5, 1, [2, 0]
    else:
        name = "g2s2" if case == "g2s2" else "g10s10"
        ds, n, burn, T, spc, chosen = S.Dataset.from_bits(*load_hex_dataset(name)), 6, 20, 77, 10, [4, 1, 5]
    run = S.Run(ds, n, seed=11, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T, manycd=manycd)
    run.init().advance(burn, False).advance(T, True).sync()
    assert (run.kernel_path() == 0) == (case not in ("big", "synthetic"))
    got = _check_run(run, chosen)
    assert got["c_sum"].shape == (len(chosen), ds.M if manycd else 1)
    _check_identity(run, got, chosen)


@pytest.mark.gpu
def test_one_shot_on_the_reference_trace(S):
    """the unmodified reference's recorded manycd run: counts over its own c, d of every sample, bit-exact"""
    g = np.load(os.path.join(GOLDEN, "ref_g10s10_manycd.npz"))
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    calls = len(g["kind"]) - 1
    run = S.Run(ds, 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls, manycd=True)
    run.set_tapes([g["tape"]]).init().advance(calls, True).sync()
    got = _check_run(run, [0])
    _compare(got, _ref(g["c_all"][1:], g["d_all"][1:]), 0, "reference trace")
    assert got["n_samples"][0] == calls
    _check_identity(run, got, [0])


def _same(x, y, what):
    for key in KEYS + ("n_samples",):
        assert x[key].tobytes() == y[key].tobytes(), (what, key)


@pytest.mark.gpu
@pytest.mark.parametrize("manycd", [False, True])
def test_streaming_equals_one_shot(S, manycd):
    ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(70), 33, 70, 3, .12))
    burn, T, chosen = 5, 70, [1, 4, 99]                     # 99: held by no run here
    kw = dict(seed=4, store=S.STORE_FULL, manycd=manycd)
    ref = S.Run(ds, 6, max_samples=T, **kw).init().advance(burn, False).advance(T, True).sync()
    want = ref.cd_marginals(chosen)
    assert want["n_samples"].tolist() == [T, T, 0]
    for W in (1, 7, 64):
        whole = S.Run(ds, 6, max_samples=W, **kw).init().accumulate(po=False, sums=False, cd=True)
        whole.advance(burn, False).advance(T, True).sync()
        _same(whole.cd_marginals(chosen), want, ("contiguous", W))
        sub = S.Run(ds, 0, max_samples=W, chain_ids=[4, 1], **kw).init().accumulate(cd=True, taxon_pairs=True)
        sub.advance_both(burn, 5).advance(T - 5, True).sync()  # 5 and 65 samples: neither a multiple of 7 or 64
        _same(sub.cd_marginals(chosen), want, ("subset", W))
        whole.close()
        sub.close()
    odd = S.Run(ds, 0, max_samples=16, chain_ids=[1, 4], **kw).init().accumulate(po=True, sums=False, cd=True)
    odd.advance_both(burn, 7).advance(20, True).advance(43, True).sync()
    _same(odd.cd_marginals(chosen), want, "advances off the window")


@pytest.mark.gpu
@pytest.mark.parametrize("manycd", [False, True])
def test_checkpoint_mid_sampling(S, tmp_path, manycd):
    """N = 33: the pair-order part is 33 * 33 words, so the cd part starts after a padding word"""
    ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(33), 33, 45, 2, .15))
    burn, T, W, chosen = 5, 50, 16, [0, 2]
    flags = dict(po=True, sums=False, cd=True)
    kw = dict(seed=8, store=S.STORE_FULL, max_samples=W, manycd=manycd)
    whole = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(T, True).sync()
    want = whole.cd_marginals(chosen)
    whole.save_checkpoint(str(tmp_path / "whole.ckpt"))
    one = S.Run(ds, 3, seed=8, store=S.STORE_FULL, max_samples=T, manycd=manycd).init().advance(burn, False).advance(T, True).sync()
    _same(one.cd_marginals(chosen), want, "one-shot")
    part = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(23, True)
    part.save_checkpoint(str(tmp_path / "part.ckpt"))
    rest = S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint(str(tmp_path / "part.ckpt")).advance(T - 23, True).sync()
    _same(rest.cd_marginals(chosen), want, "resumed")
    rest.save_checkpoint(str(tmp_path / "rest.ckpt"))
    assert (tmp_path / "rest.ckpt").read_bytes() == (tmp_path / "whole.ckpt").read_bytes()
    other = S.Run(ds, 3, **kw).accumulate(po=True, sums=False)
    _raises(S, E_STATE, other.load_checkpoint, str(tmp_path / "part.ckpt"))


@pytest.mark.gpu
@pytest.mark.parametrize("manycd", [False, True])
def test_replay_chosen_and_pooled_summary(S, manycd):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, samp, k = 64, 20, 30, 3
    runs = []
    for store in (S.STORE_FULL, S.STORE_NONE):
        run = S.Run(ds, n, seed=13, store=store, max_samples=samp, manycd=manycd).init().advance(burn, False).advance(samp, True).sync()
        runs.append(S.ChainBatch(run, burn, samp, seed=13, sweeps_per_call=10, manycd=manycd))
    one, first = runs
    chosen = S.choose_chains(one, k)
    want = one.run.cd_marginals(chosen)
    two = S.replay_chosen(first, chosen, window=16, cd=True)
    assert two.run.cfg.store == S.STORE_FULL
    _same(two.run.cd_marginals(chosen), want, "replay_chosen")
    x, y = S.cd_marginals(two, chosen), S.cd_marginals(one, chosen)
    assert x["n_samples"] == y["n_samples"] == k * samp
    R = ds.M if manycd else 1
    for name in ("c", "d"):
        pooled = want[name + "_hist"].sum(axis=0, dtype=np.int64)
        total = want[name + "_sum"][0] + want[name + "_sum"][1] + want[name + "_sum"][2]
        for key in ("mean", "quantiles", "lower", "upper", "mode", "p_mode", "counts", "sum"):
            assert np.array_equal(x[name][key], y[name][key]), (name, key)
        assert np.array_equal(x[name]["counts"], pooled) and x[name]["sum"].tobytes() == total.tobytes()
        assert x[name]["mean"].tobytes() == (total / (k * samp)).tobytes()
        q = x[name]["quantiles"]
        assert q.shape == (R, 3) and np.all((q >= 0) & (q < B)) and np.all(q[:, 0] <= q[:, 1]) and np.all(q[:, 1] <= q[:, 2])
        assert np.array_equal(q, S.hist_quantiles(pooled, (0.025, 0.5, 0.975)))
        lo, hi = BOUNDS[name]
        assert np.all(x[name]["lower"] < x[name]["upper"]) and np.all(x[name]["lower"] >= np.exp(lo) * (1 - 1e-12))
        assert np.all(x[name]["upper"] <= np.exp(hi) * (1 + 1e-12))
        assert np.all((x[name]["mean"] >= np.exp(lo) * (1 - 1e-12)) & (x[name]["mean"] <= np.exp(hi) * (1 + 1e-12)))
        assert np.array_equal(x[name]["p_mode"], pooled.max(axis=1) / (k * samp))


@pytest.mark.gpu
def test_subsets_order_and_slab_convention(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    M = ds.M
    kw = dict(seed=2, store=S.STORE_FULL, max_samples=20, manycd=True)
    full = S.Run(ds, 40, **kw).init().advance(3, False).advance(20, True).sync()
    sub = S.Run(ds, 0, chain_ids=[7, 30], **kw).init().advance(3, False).advance(20, True).sync()
    want = full.cd_marginals([7, 30])
    _same(sub.cd_marginals([7, 30]), want, "subset run")
    rev = full.cd_marginals([30, 7])
    for key in KEYS:
        assert rev[key][::-1].tobytes() == want[key].tobytes(), key
    # -1 and an unheld id leave their slabs as passed; held chains' slabs are written in full
    chosen = np.array([30, -1, 8, 7], np.int32)
    k = len(chosen)
    sums = [np.full((k, M), 7.0) for _ in range(2)]
    hists = [np.full((k, M, B), 7, np.int32) for _ in range(2)]
    n = np.full(k, 7, np.int32)
    assert S.lib().ser_run_cd_marginals(sub._h, _ptr(chosen), k, _ptr(sums[0], C.c_double), _ptr(sums[1], C.c_double), _ptr(hists[0]),
                                        _ptr(hists[1]), _ptr(n)) == 0
    assert n.tolist() == [20, 0, 0, 20]
    for o, key in zip(sums + hists, KEYS):
        assert np.all(o[1] == 7) and np.all(o[2] == 7), key
        assert o[0].tobytes() == want[key][1].tobytes() and o[3].tobytes() == want[key][0].tobytes(), key
    # every subset of the outputs
    for mask in range(1, 16):
        outs = [np.full((1, M), 7.0) if mask & 1 else None, np.full((1, M), 7.0) if mask & 2 else None,
                np.full((1, M, B), 7, np.int32) if mask & 4 else None, np.full((1, M, B), 7, np.int32) if mask & 8 else None]
        n1 = np.zeros(1, np.int32)
        assert S.lib().ser_run_cd_marginals(full._h, _ptr(np.array([7], np.int32)), 1, _ptr(outs[0], C.c_double), _ptr(outs[1], C.c_double),
                                            _ptr(outs[2]), _ptr(outs[3]), _ptr(n1)) == 0
        assert n1[0] == 20
        for o, key in zip(outs, KEYS):
            if o is not None:
                assert o[0].tobytes() == want[key][0].tobytes(), (mask, key)


def _crafted(name, rng, T, R):
    """rows at the bin and clamp edges of `name` (lo, hi, just below hi, an interior edge and the double below it, below lo, above
    hi, NaN), cycling, with uniform values in between"""
    lo, hi = BOUNDS[name]
    e1, e0 = _interior_edge(name, 1)
    e128, e127 = _interior_edge(name, 128)
    edges = [lo, hi, np.nextafter(hi, -np.inf), e1, e0, e128, e127, lo - 1.0, hi + 0.25, np.nan, np.nextafter(lo, np.inf)]
    x = rng.uniform(lo, hi, (T, R))
    for t in range(T):
        for r in range(R):
            q = (t * 5 + r) % (len(edges) + 3)
            if q < len(edges):
                x[t, r] = edges[q]
    return x


@pytest.mark.gpu
@pytest.mark.parametrize("manycd,M", [(False, 9), (True, 1), (True, 31), (True, 33), (True, 70)])
def test_crafted_stores_through_a_checkpoint(S, tmp_path, manycd, M):
    """bin and clamp edges; row-block edges in R; each chain its own T"""
    N, n, rows = 24, 4, 40
    ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(M), N, M, 3, .2))
    kw = dict(seed=5, store=S.STORE_FULL, max_samples=rows, manycd=manycd)
    f = str(tmp_path / "ck")
    S.Run(ds, n, **kw).init().advance(2, False).advance(rows, True).save_checkpoint(f).close()
    rng = np.random.default_rng(M + 100)
    own = [1, 17, 33, 40]
    R = M if manycd else 1
    crafted = {}
    for c in range(n):
        cv, dv = _crafted("c", rng, rows, R), _crafted("d", rng, rows, R)
        crafted[c] = (cv[:own[c]], dv[:own[c]])

        def edit(rec, L, cv=cv, dv=dv, t=own[c]):
            cdl = np.frombuffer(bytes(rec[L["cdl"]:L["cdl"] + 24 * rows]), np.float64).reshape(rows, 3).copy()
            if manycd:
                rec[L["cd_all"]:L["cd_all"] + 16 * rows * M] = np.stack([cv, dv], axis=1).tobytes()
                cdl[:, 0], cdl[:, 1] = cv[:, 0], dv[:, 0]
            else:
                cdl[:, 0], cdl[:, 1] = cv[:, 0], dv[:, 0]
            rec[L["cdl"]:L["cdl"] + 24 * rows] = cdl.tobytes()
            struct.pack_into("<i", rec, 156, t)
        patched = _patch_record(f, c, edit)
        open(f, "wb").write(patched)
    run = S.Run(ds, n, **kw).load_checkpoint(f)
    chosen = [3, 1, 0, 2]
    got = run.cd_marginals(chosen)
    assert got["n_samples"].tolist() == [own[g] for g in chosen]
    for c, g in enumerate(chosen):
        _compare(got, _ref(*crafted[g]), c, (M, g))
        cs, ds_ = _stored(run, g)
        assert cs.tobytes() == crafted[g][0].tobytes() and ds_.tobytes() == crafted[g][1].tobytes()
    for name in ("c", "d"):                 # the clamps and the interior edges were all hit
        h = got[name + "_hist"].sum(axis=(0, 1))
        assert h[0] > 0 and h[1] > 0 and h[127] > 0 and h[128] > 0 and h[B - 1] > 0, name
    assert run.check() == 0


@pytest.mark.gpu
def test_refusals_launch_nothing(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=8, manycd=True).init().advance(8, True).sync()
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate(ranges=True).advance(8, True).sync()
    fresh = S.Run(ds, 2, store=S.STORE_FULL, max_samples=8)
    for run, msg in ((pi_only, "SER_STORE_FULL"), (acc, "SER_ACC_CD"), (fresh, "not initialised")):
        before = run.kernel_launches()
        assert msg in _raises(S, E_STATE, run.cd_marginals, [0])
        assert run.kernel_launches() == before, msg
    assert "SER_STORE_FULL" in _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_PI, max_samples=4).init().accumulate, cd=True)
    run = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init()
    before = run.kernel_launches()
    L = S.lib()
    chosen, s, n = np.zeros(1, np.int32), np.zeros(1), np.zeros(1, np.int32)
    assert L.ser_run_cd_marginals(run._h, _ptr(chosen), 1, None, None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_cd_marginals(run._h, _ptr(chosen), 0, _ptr(s, C.c_double), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_cd_marginals(run._h, None, 1, _ptr(s, C.c_double), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_cd_marginals(run._h, _ptr(chosen), 1, _ptr(s, C.c_double), None, None, None, None) == E_ARG
    for bad in (64, 256, 1024, 512 | 64, 512 | 256):     # SER_ACC_CD is bit 512; 64, 256 and the bits above 512 are not flags
        assert L.ser_run_accumulate(run._h, bad) == E_ARG, bad
    assert run.kernel_launches() == before


def _expected_csv(S, batch, chosen, manycd):
    m = S.cd_marginals(batch, chosen)
    R = len(m["c"]["mean"])
    lines = ["taxon,c_mean,c_q025,c_median,c_q975,d_mean,d_q025,d_median,d_q975"]
    for r in range(R):
        row = [str(r) if manycd else "all"]
        for name in ("c", "d"):
            e = S.cd_bin_edges(name)
            q = m[name]["quantiles"][r]
            row += ["%.6g" % v for v in (m[name]["mean"][r], m[name]["lower"][r][0], np.exp(0.5 * (e[q[1]] + e[q[1] + 1])),
                                         m[name]["upper"][r][2])]
        lines.append(",".join(row))
    return "\n".join(lines) + "\n", m


@pytest.mark.gpu
@pytest.mark.parametrize("manycd", [False, True])
def test_cli_cd_marginals(S, tmp_path, manycd):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp = 20, 60
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "2",
            "--dataset", str(tmp_path / "g10s10.txt"), "--window", "16", "--manycd", "1" if manycd else "0"]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env, cwd=tmp_path).stdout.splitlines()
    pick = lambda lines, head: [x for x in lines if x.startswith(head)]
    out = run(["--cd-marginals", str(tmp_path / "cd.csv")])
    line = pick(out, "cd marginals:")
    assert len(line) == 1
    full = S.Run(S.Dataset.from_bits(X, hard), 64, seed=0, store=S.STORE_FULL, max_samples=samp, manycd=manycd)
    full.init().advance(burn, False).advance(samp, True).sync()
    batch = S.ChainBatch(full, burn, samp, seed=0, sweeps_per_call=10, manycd=manycd)
    chosen = S.choose_chains(batch, 2)
    assert ("chosen " + " ".join(map(str, chosen))) in pick(out, "selection:")[0]
    want, m = _expected_csv(S, batch, chosen, manycd)
    assert (tmp_path / "cd.csv").read_text() == want
    label = lambda r: ("taxon %d" % r) if manycd else "all"
    rd, rc = int(np.argmax(m["d"]["mean"])), int(np.argmax(m["c"]["mean"]))
    assert line[0] == ("cd marginals: 2 chains  %d samples  highest mean d %.6g (%s)  highest mean c %.6g (%s)"
                       % (2 * samp, m["d"]["mean"][rd], label(rd), m["c"]["mean"][rc], label(rc)))
    # one replay serves all three flags: the marginal and taxon pair files and po.csv do not change
    run(["--replay-selected", "--po", str(tmp_path / "p1.csv"), "--marginals", str(tmp_path / "P"), "--taxon-pairs", str(tmp_path / "T")])
    out2 = run(["--replay-selected", "--po", str(tmp_path / "p2.csv"), "--marginals", str(tmp_path / "Q"), "--taxon-pairs", str(tmp_path / "U"),
                "--cd-marginals", str(tmp_path / "cd2.csv")])
    assert (tmp_path / "p2.csv").read_bytes() == (tmp_path / "p1.csv").read_bytes()
    for suffix in (".sites.csv", ".taxa.csv"):
        assert (tmp_path / ("Q" + suffix)).read_bytes() == (tmp_path / ("P" + suffix)).read_bytes()
    for key in ("first", "last", "precedes", "coexist"):
        assert (tmp_path / ("U.%s.csv" % key)).read_bytes() == (tmp_path / ("T.%s.csv" % key)).read_bytes()
    assert (tmp_path / "cd2.csv").read_bytes() == (tmp_path / "cd.csv").read_bytes()
    assert pick(out2, "cd marginals:") == line
