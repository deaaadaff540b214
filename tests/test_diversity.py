"""Diversity curves on the device (ser_run_diversity, one-shot and streaming through ser_run_accumulate with SER_ACC_DIV): the posterior
of range-through richness, originations and extinctions at every position and of the richness at every site's position, checked
exactly against a numpy reference of the contract over the stored samples, the reference's recorded tape and crafted stores injected
through a checkpoint, and the contract's integer identities against ser_run_alive_counts and ser_run_marginals."""
import ctypes as C
import os
import re
import shutil
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, load_hex_dataset, random_dataset
from test_checkpoint import _layout, _patch_record

E_ARG, E_STATE = -1, -4
KEYS = ("richness", "originations", "extinctions", "site_richness")
CUH = os.path.join(ROOT, "seriation-in-paleontological-data-using-mcmc_b200", "csrc", "ser_aux_kernels.cuh")
CHUNK = int(re.search(r"#define SER_DIV_CHUNK (\d+)", open(CUH).read()).group(1))


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
def _curves(a, b, pi, N):
    """per-sample curves straight from the definitions: D, O, E [T][N] and the site row D_t(pi_t(i)) [T][N]"""
    a, b, pi = (np.asarray(x, np.int64) for x in (a, b, pi))
    p = np.arange(N)[:, None]
    D, O, E = (np.zeros((len(a), N), np.int64) for _ in range(3))
    for t in range(len(a)):
        at, bt = a[t][None, :], b[t][None, :]
        D[t] = ((at <= p) & (p < bt)).sum(axis=1)
        O[t] = ((at == p) & (p < bt)).sum(axis=1)
        E[t] = ((at < bt) & (bt == p + 1)).sum(axis=1)
    return D, O, E, np.take_along_axis(D, pi, axis=1)


def _hist(X, M):
    """[N][M + 1]: row j counts the values of column j of X [T][N]"""
    T, N = X.shape
    flat = (np.arange(N)[None, :] * (M + 1) + X).ravel()
    return np.bincount(flat, minlength=N * (M + 1)).reshape(N, M + 1)


def _ref(a, b, pi, N, M):
    return {key: _hist(X, M) for key, X in zip(KEYS, _curves(a, b, pi, N))}


def _ref_others(a, b, N, M):
    """what the identities compare with: alive [N][M] of ser_run_alive_counts (closed at b), a_hist / b_hist [M][N + 1] of
    ser_run_marginals, and z [N + 1], the empty ranges at each q"""
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    p = np.arange(N)[:, None, None]
    alive = ((a[None] <= p) & (p <= b[None])).sum(axis=1)
    a_hist = np.stack([np.bincount(a[:, m], minlength=N + 1) for m in range(M)])
    b_hist = np.stack([np.bincount(b[:, m], minlength=N + 1) for m in range(M)])
    z = np.bincount(a[a == b], minlength=N + 1)
    return alive, a_hist, b_hist, z


def _check_identities(div, T, alive, a_hist, b_hist, z):
    """the contract's exact integer identities on one chain's four outputs"""
    N, B = div["richness"].shape
    v = np.arange(B, dtype=np.int64)
    for key in KEYS:
        assert np.all(div[key].sum(axis=1) == T), key
    assert np.array_equal(div["site_richness"].sum(axis=0), div["richness"].sum(axis=0))
    s = {key: div[key].astype(np.int64) @ v for key in KEYS[:3]}
    assert np.array_equal(s["richness"], alive.sum(axis=1) - b_hist[:, :N].sum(axis=0))
    assert np.array_equal(s["originations"], a_hist[:, :N].sum(axis=0) - z[:N])
    assert np.array_equal(s["extinctions"], b_hist[:, 1:].sum(axis=0) - z[1:])
    prev = np.concatenate([[0], s["richness"][:-1]])
    prev_ext = np.concatenate([[0], s["extinctions"][:-1]])
    assert np.array_equal(s["richness"], prev + s["originations"] - prev_ext)


def _check_ref_identities(a, b, pi, N, M):
    div = _ref(a, b, pi, N, M)
    _check_identities(div, len(a), *_ref_others(a, b, N, M))
    return div


# ----------------------------------------------------------------------------- CPU
def test_reference_on_hand_written_cases():
    N, M = 5, 7
    # taxa: empty at 0, empty at 2, empty at N, all of [0, N), singleton at 0, singleton at N - 1, [1, 4)
    a = np.array([[0, 2, 5, 0, 0, 4, 1]])
    b = np.array([[0, 2, 5, 5, 1, 5, 4]])
    pi = np.array([[4, 3, 2, 1, 0]])
    D, O, E, site = _curves(a, b, pi, N)
    assert D[0].tolist() == [2, 2, 2, 2, 2]
    assert O[0].tolist() == [2, 1, 0, 0, 1]         # the whole range and a singleton start at 0, [1, 4) at 1, a singleton at 4
    assert E[0].tolist() == [1, 0, 0, 1, 2]         # the singleton at 0, [1, 4) at 3, the whole range and a singleton at 4
    assert site[0].tolist() == D[0][::-1].tolist()
    div = _check_ref_identities(a, b, pi, N, M)
    assert div["richness"][:, 2].tolist() == [1] * N and div["originations"][0, 2] == 1 and div["extinctions"][4, 2] == 1
    # every taxon alive at one position: bin M
    a, b = np.full((3, M), 2), np.full((3, M), 3)
    a[1], b[1] = 0, N                               # sample 1: every taxon over the whole sequence
    pi = np.tile(np.arange(N), (3, 1))
    div = _check_ref_identities(a, b, pi, N, M)
    assert div["richness"][2, M] == 3 and div["richness"][0, M] == 1 and div["richness"][0, 0] == 2
    assert div["originations"][2, M] == 2 and div["extinctions"][2, M] == 2 and div["originations"][0, M] == 1
    assert div["extinctions"][N - 1, M] == 1 and div["site_richness"][2, M] == 3
    # the smallest shape a run accepts, N = 2, and one taxon
    a, b = np.array([[0], [1], [0], [2], [1]]), np.array([[2], [2], [0], [2], [1]])
    pi = np.array([[0, 1], [1, 0], [0, 1], [1, 0], [0, 1]])
    div = _check_ref_identities(a, b, pi, 2, 1)
    assert div["richness"].tolist() == [[4, 1], [3, 2]]
    assert div["originations"].tolist() == [[4, 1], [4, 1]]
    assert div["extinctions"].tolist() == [[5, 0], [3, 2]]
    assert div["site_richness"].tolist() == [[3, 2], [4, 1]]


def _random_store(rng, T, N, M, empty=0.1):
    """T samples of M half-open ranges (some empty, some over the whole sequence) and T site permutations"""
    a = rng.integers(0, N + 1, (T, M))
    b = np.minimum(N, a + rng.integers(0, N + 1, (T, M)))
    e = rng.random((T, M)) < empty
    b[e] = a[e]
    w = rng.random((T, M)) < 0.05
    a[w], b[w] = 0, N
    pi = np.stack([rng.permutation(N) for _ in range(T)])
    return a, b, pi


def test_reference_identities_on_random_ranges():
    rng = np.random.default_rng(5)
    for N, M, T in ((2, 1, 9), (7, 3, 20), (33, 40, 15), (64, 9, 11)):
        a, b, pi = _random_store(rng, T, N, M)
        _check_ref_identities(a, b, pi, N, M)


def test_header_and_python_constants(S):
    text = open(os.path.join(ROOT, "include", "seriation_b200.h")).read()
    assert int(re.search(r"#define SER_ACC_DIV (\d+)", text).group(1)) == S.ACC_DIV == 2048
    assert S.DIVERSITY == KEYS
    assert "ser_run_diversity" in [s[0] for s in S.api.SYMBOLS]


def test_argument_checks_without_a_device(S):
    L = S.lib()
    chosen, out, n = np.zeros(1, np.int32), np.zeros((1, 2, 2), np.int32), np.zeros(1, np.int32)
    assert L.ser_run_diversity(None, _ptr(chosen), 1, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_accumulate(None, 2048) == E_ARG


def test_diversity_kernels_are_built_for_sm100a_without_stack_or_spills(S):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump is not installed")
    out = subprocess.run([exe, "-res-usage", S.LIB_PATH], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    lines = out.splitlines()
    for name in ("ser_div_curve_kernel", "ser_div_hist_kernel"):
        idx = [i for i, ln in enumerate(lines) if "Function" in ln and name in ln]
        assert len(idx) == 1, name
        res = lines[idx[0] + 1]
        assert "STACK:0" in res and "LOCAL:0" in res, (name, res)


def test_cli_diversity_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--diversity", str(tmp_path / "D")],
                       capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 1 and "usage" in r.stderr and "--diversity" in r.stderr
    assert not list(tmp_path.iterdir())


# ----------------------------------------------------------------------------- GPU
def _check_run(run, chosen, local=None, others=True):
    """diversity of `chosen` against the reference over each chain's fetched samples; with `others` the identities against the
    device's own alive counts and a / b histograms"""
    got = run.diversity(chosen)
    N, M = run.N, run.M
    if others:
        alive = run.alive_counts(chosen)[0]
        marg = run.marginals(chosen, ranges=True, positions=False)
    for c, g in enumerate(chosen):
        s = run.fetch_samples(g if local is None else local[c])
        T = len(s["a"])
        assert got["n_samples"][c] == T, g
        want = _ref(s["a"], s["b"], s["pi"], N, M)
        for key in KEYS:
            assert np.array_equal(got[key][c], want[key]), (g, key)
        mine = {key: got[key][c] for key in KEYS}
        _check_identities(mine, T, *_ref_others(s["a"], s["b"], N, M))
        if others:
            z = _ref_others(s["a"], s["b"], N, M)[3]
            _check_identities(mine, T, alive[c], marg["a"][c], marg["b"][c], z)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["g10s10", "g2s2", "manycd", "big", "synthetic"])
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
    got = _check_run(run, chosen, others=case != "synthetic")
    assert got["richness"].shape == (len(chosen), ds.N, ds.M + 1)


@pytest.mark.gpu
def test_one_shot_on_the_reference_tape(S):
    g = np.load(os.path.join(GOLDEN, "ref_g10s10.npz"))
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    calls = len(g["kind"]) - 1
    run = S.Run(ds, 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls).set_tapes([g["tape"]]).init().advance(calls, True).sync()
    got = _check_run(run, [0])
    assert got["n_samples"][0] == calls


def _crafted_store(rng, T, N, M):
    """random ranges with, cycling over the rows, empty ranges at 0, in the middle and at N, whole ranges, singletons at both ends, and
    every taxon at one position (bin M)"""
    a, b, pi = _random_store(rng, T, N, M)
    for t in range(T):
        q = t % 6
        if q == 0:
            a[t], b[t] = N // 2, N // 2 + 1             # every taxon alive at one position only
        elif q == 1:
            a[t], b[t] = 0, N                           # every taxon alive everywhere
        elif q == 2:
            a[t, ::3], b[t, ::3] = 0, 0
            a[t, 1::3], b[t, 1::3] = N, N
            a[t, 2::3], b[t, 2::3] = N // 2, N // 2
        elif q == 3:
            a[t, ::2], b[t, ::2] = 0, 1
            a[t, 1::2], b[t, 1::2] = N - 1, N
    return a.astype(np.uint16), b.astype(np.uint16), pi.astype(np.uint16)


def _inject(S, ds, tmp_path, n, rows, own, seed):
    """a STORE_FULL checkpoint of n chains holding `rows` rows each, with crafted a, b and pi rows and each chain's own T"""
    N, M = ds.N, ds.M
    kw = dict(seed=5, store=S.STORE_FULL, max_samples=rows)
    f = str(tmp_path / "ck")
    S.Run(ds, n, **kw).init().advance(2, False).advance(rows, True).save_checkpoint(f).close()
    assert _layout(N, M, 0, S.STORE_FULL, rows, 0)["size"] == struct.unpack_from("<Q", open(f, "rb").read(104), 88)[0]
    rng = np.random.default_rng(seed)
    crafted = {}
    for c in range(n):
        a, b, pi = _crafted_store(rng, rows, N, M)
        crafted[c] = (a[:own[c]], b[:own[c]], pi[:own[c]])

        def edit(rec, L, a=a, b=b, pi=pi, t=own[c]):
            rec[L["sa"]:L["sa"] + a.nbytes] = a.tobytes()
            rec[L["sb"]:L["sb"] + b.nbytes] = b.tobytes()
            rec[L["spi"]:L["spi"] + pi.nbytes] = pi.tobytes()
            struct.pack_into("<i", rec, 156, t)
        patched = _patch_record(f, c, edit)
        open(f, "wb").write(patched)
    return S.Run(ds, n, **kw).load_checkpoint(f), crafted


def _check_crafted(run, crafted, chosen):
    got = run.diversity(chosen)
    N, M = run.N, run.M
    assert got["n_samples"].tolist() == [len(crafted[g][0]) for g in chosen]
    for c, g in enumerate(chosen):
        a, b, pi = crafted[g]
        s = run.fetch_samples(g)
        assert np.array_equal(s["a"], a) and np.array_equal(s["b"], b) and np.array_equal(s["pi"], pi)
        want = _ref(a, b, pi, N, M)
        for key in KEYS:
            assert np.array_equal(got[key][c], want[key]), (N, M, g, key)
        _check_identities({key: got[key][c] for key in KEYS}, len(a), *_ref_others(a, b, N, M))
    return got


# stage 1 scans 256 positions at a time; stage 2 gives a block 128 rows while (M + 1) * 128 ints fit 96 KiB, 64 or 32 rows when they fit
# that way, and counts in global memory from M + 1 = 769 on
@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(31, 1), (32, 31), (33, 32), (64, 33), (65, 191), (128, 192), (129, 255), (255, 256), (256, 383),
                                 (257, 384), (300, 767), (40, 768), (513, 1000)])
def test_crafted_stores_through_a_checkpoint(S, tmp_path, N, M):
    ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(N * M), N, M, 3, .15))
    own = [1, 12, 30, 40]
    run, crafted = _inject(S, ds, tmp_path, 4, 40, own, N + M)
    got = _check_crafted(run, crafted, [3, 1, 0, 2])
    assert got["richness"][:, :, M].sum() > 0 and got["site_richness"][:, :, M].sum() > 0    # bin M was hit
    assert run.check() == 0


@pytest.mark.gpu
def test_crafted_stores_at_the_pass_edges(S, tmp_path):
    """each chain its own T around the one-shot getter's pass of SER_DIV_CHUNK rows"""
    ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(9), 40, 20, 3, .15))
    own = [CHUNK - 1, CHUNK, CHUNK + 1, 3]
    run, crafted = _inject(S, ds, tmp_path, 4, CHUNK + 1, own, 77)
    _check_crafted(run, crafted, [2, 0, 1, 3])
    _check_crafted(run, crafted, [0])          # a getter whose chain's T is one pass


@pytest.mark.gpu
def test_subsets_order_and_slab_convention(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    N, M = ds.N, ds.M
    kw = dict(seed=2, store=S.STORE_FULL, max_samples=20)
    full = S.Run(ds, 40, **kw).init().advance(3, False).advance(20, True).sync()
    sub = S.Run(ds, 0, chain_ids=[7, 30], **kw).init().advance(3, False).advance(20, True).sync()
    want = full.diversity([7, 30])
    _same(sub.diversity([7, 30]), want, "subset run")
    rev = full.diversity([30, 7])
    for key in KEYS:
        assert rev[key][::-1].tobytes() == want[key].tobytes(), key
    # -1 and an unheld id leave their slabs as passed; held chains' slabs are written in full
    chosen = np.array([30, -1, 8, 7], np.int32)
    k = len(chosen)
    outs = [np.full((k, N, M + 1), 7, np.int32) for _ in KEYS]
    n = np.full(k, 7, np.int32)
    assert S.lib().ser_run_diversity(sub._h, _ptr(chosen), k, *(_ptr(o) for o in outs), _ptr(n)) == 0
    assert n.tolist() == [20, 0, 0, 20]
    for o, key in zip(outs, KEYS):
        assert np.all(o[1] == 7) and np.all(o[2] == 7), key
        assert o[0].tobytes() == want[key][1].tobytes() and o[3].tobytes() == want[key][0].tobytes(), key
    # every subset of the outputs
    for mask in range(1, 16):
        outs = [np.full((1, N, M + 1), 7, np.int32) if mask >> q & 1 else None for q in range(4)]
        n1 = np.zeros(1, np.int32)
        assert S.lib().ser_run_diversity(full._h, _ptr(np.array([7], np.int32)), 1, *(_ptr(o) for o in outs), _ptr(n1)) == 0
        assert n1[0] == 20
        for o, key in zip(outs, KEYS):
            if o is not None:
                assert o[0].tobytes() == want[key][0].tobytes(), (mask, key)


def _same(x, y, what):
    for key in KEYS + ("n_samples",):
        assert x[key].tobytes() == y[key].tobytes(), (what, key)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["g10s10", "33x70"])
def test_streaming_equals_one_shot(S, shape):
    if shape == "g10s10":
        ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    else:
        ds = S.Dataset.from_bits(*random_dataset(np.random.default_rng(70), 33, 70, 3, .12))
    burn, T, chosen = 5, 70, [1, 4, 99]                     # 99: held by no run here
    kw = dict(seed=4, store=S.STORE_FULL)
    ref = S.Run(ds, 6, max_samples=T, **kw).init().advance(burn, False).advance(T, True).sync()
    want = ref.diversity(chosen)
    assert want["n_samples"].tolist() == [T, T, 0]
    for W in (1, 7, 64):
        whole = S.Run(ds, 6, max_samples=W, **kw).init().accumulate(po=False, sums=False, diversity=True)
        whole.advance(burn, False).advance(T, True).sync()
        _same(whole.diversity(chosen), want, ("contiguous", W))
        sub = S.Run(ds, 0, max_samples=W, chain_ids=[4, 1], **kw).init().accumulate(diversity=True, cd=True)
        sub.advance_both(burn, 5).advance(T - 5, True).sync()  # 5 and 65 samples: neither a multiple of 7 or 64
        _same(sub.diversity(chosen), want, ("subset", W))
        whole.close()
        sub.close()
    odd = S.Run(ds, 0, max_samples=16, chain_ids=[1, 4], **kw).init().accumulate(po=True, sums=False, diversity=True)
    odd.advance_both(burn, 7).advance(20, True).advance(43, True).sync()
    _same(odd.diversity(chosen), want, "advances off the window")


@pytest.mark.gpu
def test_replay_chosen_and_pooled_summary(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, samp, k = 64, 20, 30, 3
    one = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_FULL)
    chosen = S.choose_chains(one, k)
    want = one.run.diversity(chosen)
    first = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_NONE)
    two = S.replay_chosen(first, chosen, window=16, diversity=True)
    assert two.run.cfg.store == S.STORE_FULL
    _same(two.run.diversity(chosen), want, "replay_chosen")
    x, y = S.diversity(two, chosen), S.diversity(one, chosen)
    assert x["n_samples"] == y["n_samples"] == k * samp
    v = np.arange(ds.M + 1)
    for key in KEYS:
        pooled = want[key].sum(axis=0, dtype=np.int64)
        assert np.array_equal(x["counts"][key], pooled) and np.array_equal(y["counts"][key], pooled), key
        for f in ("mean", "quantiles", "mode", "p_mode"):
            assert np.array_equal(x[key][f], y[key][f]), (key, f)
        assert np.array_equal(x[key]["mean"], (pooled @ v) / (k * samp)), key
        q = x[key]["quantiles"]
        assert q.shape == (ds.N, 3) and np.all(q[:, 0] <= q[:, 1]) and np.all(q[:, 1] <= q[:, 2]) and np.all((q >= 0) & (q <= ds.M))
        assert np.array_equal(q, S.hist_quantiles(pooled, (0.025, 0.5, 0.975))), key
        assert np.array_equal(x[key]["p_mode"], pooled.max(axis=1) / (k * samp)), key


@pytest.mark.gpu
def test_checkpoint_mid_window(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    burn, T, W, chosen = 5, 50, 16, [0, 2]
    flags = dict(po=True, sums=False, cd=True, diversity=True)
    kw = dict(seed=8, store=S.STORE_FULL, max_samples=W)
    whole = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(T, True).sync()
    want = whole.diversity(chosen)
    whole.save_checkpoint(str(tmp_path / "whole.ckpt"))
    one = S.Run(ds, 3, seed=8, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    _same(one.diversity(chosen), want, "one-shot")
    part = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(23, True)
    part.save_checkpoint(str(tmp_path / "part.ckpt"))
    rest = S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint(str(tmp_path / "part.ckpt")).advance(T - 23, True).sync()
    _same(rest.diversity(chosen), want, "resumed")
    rest.save_checkpoint(str(tmp_path / "rest.ckpt"))
    assert (tmp_path / "rest.ckpt").read_bytes() == (tmp_path / "whole.ckpt").read_bytes()
    # a run accumulating other flags does not load it, and neither does one that adds the flag to a file without it
    _raises(S, E_STATE, S.Run(ds, 3, **kw).accumulate(po=True, sums=False, cd=True).load_checkpoint, str(tmp_path / "part.ckpt"))
    plain = S.Run(ds, 3, **kw).init().accumulate(po=True, sums=False, cd=True).advance(burn, False).advance(9, True)
    plain.save_checkpoint(str(tmp_path / "plain.ckpt"))
    _raises(S, E_STATE, S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint, str(tmp_path / "plain.ckpt"))


@pytest.mark.gpu
def test_checkpoint_record_above_the_staging_size(S, tmp_path):
    """at 1024 x 4096 the diversity part is 67 MB and the taxon pair part 256 MiB: one record is larger than the 256 MiB a save or load
    stages through"""
    ds = S.Dataset.synthetic(1024, 4096, 16)
    kw = dict(seed=9, sweeps_per_call=1, store=S.STORE_FULL, max_samples=4, chain_ids=[5])
    flags = dict(po=False, sums=False, taxon_pairs=True, diversity=True)
    whole = S.Run(ds, 0, **kw).init().accumulate(**flags).advance(1, False).advance(9, True).sync()
    want = whole.diversity([5])
    whole.close()
    f = str(tmp_path / "big.ckpt")
    S.Run(ds, 0, **kw).init().accumulate(**flags).advance(1, False).advance(6, True).save_checkpoint(f).close()
    size = struct.unpack_from("<Q", open(f, "rb").read(104), 88)[0]
    assert size > 256 << 20
    rest = S.Run(ds, 0, **kw).accumulate(**flags).load_checkpoint(f).advance(3, True).sync()
    _same(rest.diversity([5]), want, "resumed large record")
    assert want["n_samples"].tolist() == [9]


@pytest.mark.gpu
def test_same_batch_twice_gives_the_same_bytes(S):
    ds = S.Dataset.synthetic(256, 700, 8)
    outs = []
    for _ in range(2):
        run = S.Run(ds, 3, seed=21, sweeps_per_call=2, store=S.STORE_FULL, max_samples=40).init().advance(3, False).advance(40, True).sync()
        outs.append(run.diversity([2, 0, 1]))
        outs.append(run.diversity([2, 0, 1]))
        run.close()
    for o in outs[1:]:
        _same(o, outs[0], "repeat")


@pytest.mark.gpu
def test_refusals_launch_nothing(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=8).init().advance(8, True).sync()
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate(ranges=True, cd=True).advance(8, True).sync()
    fresh = S.Run(ds, 2, store=S.STORE_FULL, max_samples=8)
    for run, msg in ((pi_only, "SER_STORE_FULL"), (acc, "SER_ACC_DIV"), (fresh, "not initialised")):
        before = run.kernel_launches()
        assert msg in _raises(S, E_STATE, run.diversity, [0])
        assert run.kernel_launches() == before, msg
    assert "SER_STORE_FULL" in _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_PI, max_samples=4).init().accumulate, diversity=True)
    run = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init()
    before = run.kernel_launches()
    L = S.lib()
    chosen, out, n = np.zeros(1, np.int32), np.zeros((1, ds.N, ds.M + 1), np.int32), np.zeros(1, np.int32)
    assert L.ser_run_diversity(run._h, _ptr(chosen), 1, None, None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_diversity(run._h, _ptr(chosen), 0, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_diversity(run._h, None, 1, _ptr(out), None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_diversity(run._h, _ptr(chosen), 1, None, None, None, _ptr(out), None) == E_ARG
    for bad in (1024, 4096, 2048 | 1024, 2048 | 64):        # SER_ACC_DIV is bit 2048; 1024 and the bits above 2048 are not flags
        assert L.ser_run_accumulate(run._h, bad) == E_ARG, bad
    assert run.kernel_launches() == before


def _expected_csv(S, batch, chosen, hard):
    m = S.diversity(batch, chosen)
    N = len(hard)
    pos = ["position,rich_mean,rich_q025,rich_median,rich_q975,orig_mean,orig_q025,orig_median,orig_q975,ext_mean,ext_q025,ext_median,"
           "ext_q975"]
    for p in range(N):
        row = [str(p)]
        for key in KEYS[:3]:
            q = m[key]["quantiles"][p]
            row += ["%.6f" % m[key]["mean"][p], "%d" % q[0], "%d" % q[1], "%d" % q[2]]
        pos.append(",".join(row))
    sites = ["site,hard,rich_mean,rich_q025,rich_median,rich_q975"]
    for i in range(N):
        q = m["site_richness"]["quantiles"][i]
        sites.append("%d,%d,%.6f,%d,%d,%d" % (i, hard[i] != 0, m["site_richness"]["mean"][i], q[0], q[1], q[2]))
    return "\n".join(pos) + "\n", "\n".join(sites) + "\n", m


@pytest.mark.gpu
def test_cli_diversity(S, tmp_path):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp = 20, 60
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "2",
            "--dataset", str(tmp_path / "g10s10.txt"), "--window", "16"]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env, cwd=tmp_path).stdout.splitlines()
    pick = lambda lines, head: [x for x in lines if x.startswith(head)]
    out = run(["--diversity", str(tmp_path / "D")])
    line = pick(out, "diversity:")
    assert len(line) == 1
    full = S.Run(S.Dataset.from_bits(X, hard), 64, seed=0, store=S.STORE_FULL, max_samples=samp)
    full.init().advance(burn, False).advance(samp, True).sync()
    batch = S.ChainBatch(full, burn, samp, seed=0, sweeps_per_call=10)
    chosen = S.choose_chains(batch, 2)
    assert ("chosen " + " ".join(map(str, chosen))) in pick(out, "selection:")[0]
    want_pos, want_sites, m = _expected_csv(S, batch, chosen, hard)
    assert (tmp_path / "D.positions.csv").read_text() == want_pos
    assert (tmp_path / "D.sites.csv").read_text() == want_sites
    r = m["richness"]
    peak = int(np.argmax(r["mean"]))
    assert line[0] == ("diversity: 2 chains  %d samples  peak mean richness %.6f taxa at position %d (95%% interval %d-%d)"
                       % (2 * samp, r["mean"][peak], peak, r["quantiles"][peak][0], r["quantiles"][peak][2]))
    # one replay serves every flag: the other outputs do not change with --diversity, with the window and with the full store
    others = ["--replay-selected", "--po", "p.csv", "--marginals", "P", "--taxon-pairs", "T", "--cd-marginals", "cd.csv"]
    files = ["p.csv", "P.sites.csv", "P.taxa.csv", "T.first.csv", "T.last.csv", "T.precedes.csv", "T.coexist.csv", "cd.csv"]
    for extra in ([], ["--diagnostics", "diag.csv"]):
        results = []
        for div in ([], ["--diversity", "E"]):
            for name in files:
                (tmp_path / name).unlink(missing_ok=True)
            lines = run(others + extra + div)
            results.append(({name: (tmp_path / name).read_bytes() for name in files}, [x for x in lines if not x.startswith("diversity:")]))
            if div:
                assert pick(lines, "diversity:") == line, extra
                assert (tmp_path / "E.positions.csv").read_bytes() == (tmp_path / "D.positions.csv").read_bytes(), extra
                assert (tmp_path / "E.sites.csv").read_bytes() == (tmp_path / "D.sites.csv").read_bytes(), extra
        assert results[0][0] == results[1][0], extra
        strip = lambda lines: [x for x in lines if not x.startswith("chains ")]    # the timing line
        assert strip(results[0][1]) == strip(results[1][1]), extra
