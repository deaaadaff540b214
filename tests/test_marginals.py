"""Posterior marginals: per-site position and per-taxon a / b histograms on the device (ser_run_marginals, one-shot and streaming
through ser_run_accumulate), their quantiles on the host (ser_hist_quantiles), checked against np.add.at over the stored samples."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, load_hex_dataset

E_ARG, E_STATE = -1, -4
i32p, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)


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


# ----------------------------------------------------------------------------- CPU
def _ref_quantiles(h, probs):
    cum = np.cumsum(h.astype(np.int64), axis=1)
    out = np.empty((h.shape[0], len(probs)), np.int32)
    for r in range(h.shape[0]):
        out[r] = -1 if cum[r, -1] == 0 else [np.searchsorted(cum[r], p * cum[r, -1], side="left") for p in probs]
    return out


def test_hist_quantiles_equal_numpy(S):
    rng = np.random.default_rng(5)
    probs = (0.025, 0.1, 0.5, 0.9, 0.975, 1.0)
    for rows, bins in ((1, 1), (7, 2), (50, 125), (20, 2049)):
        h = rng.integers(0, 4, (rows, bins)).astype(np.int32) * (rng.random((rows, bins)) < 0.2)
        h[0] = 0                                          # an empty row
        if rows > 1:
            h[1] = 0
            h[1, rng.integers(bins)] = 1000               # all mass in one bin
        got = S.hist_quantiles(h, probs)
        assert np.array_equal(got, _ref_quantiles(h, probs)), (rows, bins)
        assert np.all(got[0] == -1)
    # p * T exactly an integer: the median of T = 1000 is the first bin whose count reaches 500
    h = np.zeros((1, 10), np.int32)
    h[0, 3], h[0, 7] = 500, 500
    assert S.hist_quantiles(h, [0.5, 0.5000001, 1.0]).tolist() == [[3, 7, 7]]
    # leading dimensions are kept
    h3 = rng.integers(0, 5, (2, 3, 11)).astype(np.int32)
    assert S.hist_quantiles(h3, [0.5]).shape == (2, 3, 1)
    assert np.array_equal(S.hist_quantiles(h3, [0.5])[..., 0], _ref_quantiles(h3.reshape(6, 11), [0.5]).reshape(2, 3))


def test_hist_quantiles_refusals(S):
    L = S.lib()
    h, out, probs = np.ones((2, 5), np.int32), np.zeros(4, np.int32), np.array([0.5])
    assert L.ser_hist_quantiles(_ptr(h), 0, 5, _ptr(probs, C.c_double), 1, _ptr(out)) == E_ARG
    assert L.ser_hist_quantiles(_ptr(h), 2, 0, _ptr(probs, C.c_double), 1, _ptr(out)) == E_ARG
    assert L.ser_hist_quantiles(None, 2, 5, _ptr(probs, C.c_double), 1, _ptr(out)) == E_ARG
    assert L.ser_hist_quantiles(_ptr(h), 2, 5, None, 1, _ptr(out)) == E_ARG
    assert L.ser_hist_quantiles(_ptr(h), 2, 5, _ptr(probs, C.c_double), 1, None) == E_ARG
    for bad in (0.0, -0.5, 1.0000001, 2.0, np.nan):
        p = np.array([0.5, bad])
        assert L.ser_hist_quantiles(_ptr(h), 2, 5, _ptr(p, C.c_double), 2, _ptr(out)) == E_ARG, bad
        assert b"is not in (0, 1]" in L.ser_last_error()


def test_marginals_argument_checks_without_a_device(S):
    L = S.lib()
    chosen, pos, n = np.zeros(1, np.int32), np.zeros(64, np.int32), np.zeros(1, np.int32)
    for k, p, nn in ((1, pos, n), (0, pos, n), (1, None, n), (1, pos, None)):
        assert L.ser_run_marginals(None, _ptr(chosen), k, _ptr(p), None, None, _ptr(nn)) == E_ARG
    assert L.ser_run_accumulate(None, 64) == E_ARG
    assert L.ser_run_accumulate(None, 16 | 32) == E_ARG


def test_summary_kernels_are_built_for_sm100a_without_stack_or_spills(S):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(exe):
        pytest.skip("cuobjdump is not installed")
    out = subprocess.run([exe, "-res-usage", S.LIB_PATH], check=True, capture_output=True, text=True).stdout
    assert "sm_100a" in out
    names = ("ser_po_kernel", "ser_posterior_kernel", "ser_alive_kernel", "ser_pos_hist_kernel", "ser_range_hist_kernel",
             "ser_po_acc_out_kernel", "ser_posterior_acc_out_kernel", "ser_alive_acc_out_kernel", "ser_hist_acc_out_kernel",
             "ser_diag_kernel")
    lines = out.splitlines()
    for name in names:
        idx = [i for i, ln in enumerate(lines) if "Function" in ln and name in ln]
        assert len(idx) == 1, name
        res = lines[idx[0] + 1]
        assert "STACK:0" in res and "LOCAL:0" in res, (name, res)


def test_cli_marginals_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--marginals", str(tmp_path / "m")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "usage" in r.stderr and not (tmp_path / "m.sites.csv").exists()


# ----------------------------------------------------------------------------- GPU
def _ref(run, g):
    """np.add.at over the stored samples of chain g (local index = global on the runs used with it)"""
    s = run.fetch_samples(g)
    T, N, M = s["pi"].shape[0], run.N, run.M
    pos, a, b = np.zeros((N, N), np.int32), np.zeros((M, N + 1), np.int32), np.zeros((M, N + 1), np.int32)
    np.add.at(pos, (np.tile(np.arange(N), T), s["pi"].ravel()), 1)
    np.add.at(a, (np.tile(np.arange(M), T), s["a"].ravel()), 1)
    np.add.at(b, (np.tile(np.arange(M), T), s["b"].ravel()), 1)
    return pos, a, b, T


def _check_one_shot(S, run, chosen, local=None):
    m = run.marginals(chosen, ranges=True)
    ps = run.posterior_sums(chosen, with_ab=True)
    N, M = run.N, run.M
    for c, g in enumerate(chosen):
        pos, a, b, T = _ref(run, g if local is None else local[c])
        assert m["n_samples"][c] == T
        assert np.array_equal(m["pos"][c], pos) and np.array_equal(m["a"][c], a) and np.array_equal(m["b"][c], b), g
        assert np.all(m["pos"][c].sum(axis=1) == T) and np.all(m["a"][c].sum(axis=1) == T) and np.all(m["b"][c].sum(axis=1) == T)
        assert np.array_equal(m["pos"][c].astype(np.int64) @ np.arange(N), ps["pi_sum"][c])
        assert np.array_equal(m["a"][c].astype(np.int64) @ np.arange(N + 1), ps["a_sum"][c])
        assert np.array_equal(m["b"][c].astype(np.int64) @ np.arange(N + 1), ps["b_sum"][c])
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["g2s2", "synthetic", "manycd"])
def test_one_shot_equals_numpy(S, case):
    if case == "synthetic":
        ds, n, burn, T, spc, chosen = S.Dataset.synthetic(1024, 4096, 16), 3, 2, 30, 1, [2, 0]
    else:
        ds, n, burn, T, spc, chosen = S.Dataset.from_bits(*load_hex_dataset("g2s2" if case == "g2s2" else "g10s10")), 6, 20, 120, 10, [4, 1, 5]
    run = S.Run(ds, n, seed=11, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T, manycd=case == "manycd")
    run.init().advance(burn, False).advance(T, True).sync()
    assert (run.kernel_path() == 0) == (case != "synthetic")   # the one-thread-per-taxon kernel, or the large-shape kernel
    _check_one_shot(S, run, chosen)


@pytest.mark.gpu
def test_one_shot_on_the_reference_tape(S):
    g = np.load(os.path.join(GOLDEN, "ref_g10s10.npz"))
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    calls = len(g["kind"]) - 1
    run = S.Run(ds, 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls).set_tapes([g["tape"]]).init().advance(calls, True).sync()
    m = _check_one_shot(S, run, [0])
    assert m["n_samples"][0] == calls
    # the last sample of the reference's own trace is among the counted ones
    assert np.all(m["pos"][0][np.arange(ds.N), g["pi"][-1].astype(np.int64)] >= 1)


@pytest.mark.gpu
def test_slab_convention(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    N, M = ds.N, ds.M
    run = S.Run(ds, 0, seed=2, store=S.STORE_FULL, max_samples=20, chain_ids=[7, 30]).init().advance(3, False).advance(20, True).sync()
    want = run.marginals([7, 30], ranges=True)
    chosen = np.array([30, -1, 8, 7], np.int32)
    k = len(chosen)
    pos, a, b = np.full((k, N, N), 7, np.int32), np.full((k, M, N + 1), 7, np.int32), np.full((k, M, N + 1), 7, np.int32)
    n = np.full(k, 7, np.int32)
    assert S.lib().ser_run_marginals(run._h, _ptr(chosen), k, _ptr(pos), _ptr(a), _ptr(b), _ptr(n)) == 0
    assert n.tolist() == [20, 0, 0, 20]
    for c in (1, 2):
        assert np.all(pos[c] == 7) and np.all(a[c] == 7) and np.all(b[c] == 7)
    for c, w in ((0, 1), (3, 0)):
        assert np.array_equal(pos[c], want["pos"][w]) and np.array_equal(a[c], want["a"][w]) and np.array_equal(b[c], want["b"][w])
    # one output alone; the others stay untouched
    pos2, n2 = np.full((1, N, N), 7, np.int32), np.zeros(1, np.int32)
    assert S.lib().ser_run_marginals(run._h, _ptr(np.array([7], np.int32)), 1, _ptr(pos2), None, None, _ptr(n2)) == 0
    assert np.array_equal(pos2[0], want["pos"][0]) and n2[0] == 20


def _same(x, y, what):
    for key in ("pos", "a", "b", "n_samples"):
        assert np.array_equal(x[key], y[key]), (what, key)


@pytest.mark.gpu
def test_streaming_equals_one_shot(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    burn, T, chosen = 5, 70, [1, 4, 99]                  # 99: held by no run here
    ref = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    want = ref.marginals(chosen, ranges=True)
    assert want["n_samples"].tolist() == [T, T, 0]
    for W in (1, 3, 16, 64):
        whole = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=W).init().accumulate(po=False, sums=False, positions=True, ranges=True)
        whole.advance(burn, False).advance(T, True).sync()
        _same(whole.marginals(chosen, ranges=True), want, ("contiguous", W))
        sub = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=W, chain_ids=[4, 1]).init().accumulate(positions=True, ranges=True)
        sub.advance(burn, False).advance(T, True).sync()
        _same(sub.marginals(chosen, ranges=True), want, ("subset", W))
    odd = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=16, chain_ids=[1, 4]).init().accumulate(positions=True, ranges=True)
    odd.advance_both(burn, 7).advance(20, True).advance(43, True).sync()
    _same(odd.marginals(chosen, ranges=True), want, "advances off the window")
    # positions alone through a pi-only window
    pi = S.Run(ds, 6, seed=4, store=S.STORE_PI, max_samples=9).init().accumulate(po=False, sums=False, positions=True)
    pi.advance(burn, False).advance(T, True).sync()
    got = pi.marginals(chosen)
    assert np.array_equal(got["pos"], want["pos"]) and got["a"] is None


@pytest.mark.gpu
def test_more_samples_than_the_window_holds_on_the_large_shape(S):
    ds = S.Dataset.synthetic(1024, 4096, 16)
    seed, burn, T = 20060206, 2, 40
    sub = S.Run(ds, 0, seed=seed, sweeps_per_call=1, store=S.STORE_FULL, max_samples=8, chain_ids=[3, 40000]).init()
    sub.accumulate(po=False, sums=False, positions=True, ranges=True).advance(burn, False).advance(T, True).sync()
    got = sub.marginals([3, 40000], ranges=True)
    for c, g in enumerate((3, 40000)):
        one = S.Run(ds, 1, seed=seed, sweeps_per_call=1, chain_offset=g, store=S.STORE_FULL, max_samples=T).init()
        one.advance(burn, False).advance(T, True).sync()
        w = _check_one_shot(S, one, [g], local=[0])
        for key in ("pos", "a", "b"):
            assert np.array_equal(got[key][c], w[key][0]), (g, key)
        assert got["n_samples"][c] == T
        one.close()


@pytest.mark.gpu
def test_subset_run_and_replay_chosen(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, samp, k = 64, 20, 30, 3
    one = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_FULL)
    chosen = S.choose_chains(one, k)
    want = one.run.marginals(chosen, ranges=True)
    sub = S.Run(ds, 0, seed=13, store=S.STORE_FULL, max_samples=samp, chain_ids=chosen[::-1]).init()
    sub.advance(burn, False).advance(samp, True).sync()
    _same(sub.marginals(chosen, ranges=True), want, "subset run")
    first = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_NONE)
    two = S.replay_chosen(first, chosen, window=16, marginals=True)
    assert two.run.cfg.store == S.STORE_FULL
    _same(two.run.marginals(chosen, ranges=True), want, "replay_chosen")
    x, y = S.marginals(two, chosen), S.marginals(one, chosen)
    for part in ("sites", "a", "b"):
        for key in ("mean", "quantiles", "mode", "p_mode"):
            assert np.array_equal(x[part][key], y[part][key]), (part, key)
    assert x["n_samples"] == k * samp
    pooled = want["pos"].sum(axis=0)
    assert np.array_equal(x["counts"]["pos"], pooled)
    assert np.array_equal(x["sites"]["quantiles"], _ref_quantiles(pooled, (0.025, 0.5, 0.975)))
    assert np.array_equal(x["sites"]["mean"], (pooled.astype(np.int64) @ np.arange(ds.N)) / (k * samp))
    assert np.array_equal(S.compute_pair_order_matrix(two, chosen, k), S.compute_pair_order_matrix(one, chosen, k))


@pytest.mark.gpu
def test_multi_device_slabs_sum_to_one_device(S):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, T, chosen = 64, 10, 25, [3, 40, 63]
    one = S.Run(ds, n, seed=6, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    want = one.marginals(chosen, ranges=True)
    m = S.Multi(ds, n, 2, seed=6, store=S.STORE_FULL, max_samples=T).init().advance(burn, T).sync()
    runs = {}
    for g in chosen:
        r, _ = m.locate(g)
        runs[r._h.value] = r
    assert len(runs) == 2
    parts = [r.marginals(chosen, ranges=True) for r in runs.values()]
    got = {key: sum(p[key] for p in parts) for key in ("pos", "a", "b", "n_samples")}
    _same(got, want, "ser_multi over 2 GPUs")


@pytest.mark.gpu
def test_checkpoint_mid_window(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    burn, T, W, chosen = 5, 50, 16, [0, 2]
    flags = dict(po=True, sums=False, alive=True, positions=True, ranges=True)
    kw = dict(seed=8, store=S.STORE_FULL, max_samples=W)
    whole = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(T, True).sync()
    want = whole.marginals(chosen, ranges=True)
    whole.save_checkpoint(str(tmp_path / "whole.ckpt"))
    part = S.Run(ds, 3, **kw).init().accumulate(**flags).advance(burn, False).advance(23, True)
    part.save_checkpoint(str(tmp_path / "part.ckpt"))
    rest = S.Run(ds, 3, **kw).accumulate(**flags).load_checkpoint(str(tmp_path / "part.ckpt")).advance(T - 23, True).sync()
    _same(rest.marginals(chosen, ranges=True), want, "resumed")
    assert np.array_equal(rest.po_counts(chosen), whole.po_counts(chosen))
    rest.save_checkpoint(str(tmp_path / "rest.ckpt"))
    assert (tmp_path / "rest.ckpt").read_bytes() == (tmp_path / "whole.ckpt").read_bytes()
    # a run accumulating other flags does not load it
    other = S.Run(ds, 3, **kw).accumulate(po=True, sums=False, alive=True)
    _raises(S, E_STATE, other.load_checkpoint, str(tmp_path / "part.ckpt"))


@pytest.mark.gpu
def test_refusals_launch_nothing(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=8).init().advance(8, True).sync()
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate(ab=True, alive=True).advance(8, True).sync()
    fresh = S.Run(ds, 2, store=S.STORE_FULL, max_samples=8)
    cases = ((pi_only, dict(ranges=True), "SER_STORE_FULL"), (acc, {}, "SER_ACC_POS"), (acc, dict(ranges=True, positions=False), "SER_ACC_RANGE"),
             (fresh, {}, "not initialised"))
    for run, kw, msg in cases:
        before = run.kernel_launches()
        assert msg in _raises(S, E_STATE, run.marginals, [0], **kw)
        assert run.kernel_launches() == before, msg
    assert "SER_STORE_FULL" in _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_PI, max_samples=4).init().accumulate, ranges=True)
    run = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init()
    before = run.kernel_launches()
    L = S.lib()
    chosen, pos, n = np.zeros(1, np.int32), np.zeros((1, ds.N, ds.N), np.int32), np.zeros(1, np.int32)
    assert L.ser_run_accumulate(run._h, 64) == E_ARG
    assert L.ser_run_marginals(run._h, _ptr(chosen), 1, None, None, None, _ptr(n)) == E_ARG
    assert L.ser_run_marginals(run._h, _ptr(chosen), 0, _ptr(pos), None, None, _ptr(n)) == E_ARG
    assert L.ser_run_marginals(run._h, _ptr(chosen), 1, _ptr(pos), None, None, None) == E_ARG
    assert run.kernel_launches() == before


def _csv(path):
    lines = open(path).read().splitlines()
    return lines[0], [ln.split(",") for ln in lines[1:]]


@pytest.mark.gpu
def test_cli_marginals(S, tmp_path):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp = 20, 60
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "2",
            "--dataset", str(tmp_path / "g10s10.txt")]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env, cwd=tmp_path).stdout.splitlines()
    plain = run([])
    out = run(["--marginals", str(tmp_path / "P")])
    pick = lambda lines, head: [x for x in lines if x.startswith(head)]
    assert pick(out, "selection:") == pick(plain, "selection:") and len(pick(out, "selection:")) == 1
    line = pick(out, "marginals:")
    assert len(line) == 1 and "median width" in line[0] and not pick(plain, "marginals:")
    batch = S.run_all_chains(S.Dataset.from_bits(X, hard), 64, burn, samp, seed=0, store=S.STORE_FULL)
    chosen = S.choose_chains(batch, 2)
    assert ("chosen " + " ".join(map(str, chosen))) in pick(out, "selection:")[0]
    mg = S.marginals(batch, chosen)
    head, rows = _csv(tmp_path / "P.sites.csv")
    assert head == "site,hard,mean,q025,median,q975,mode,p_mode" and len(rows) == X.shape[0]
    s = mg["sites"]
    for i, r in enumerate(rows):
        assert [int(v) for v in (r[0], r[1], r[3], r[4], r[5], r[6])] == [i, int(hard[i]), *s["quantiles"][i], s["mode"][i]], i
        assert r[2] == "%.6f" % s["mean"][i] and r[7] == "%.6f" % s["p_mode"][i], i
    head, rows = _csv(tmp_path / "P.taxa.csv")
    assert head == "taxon,a_mean,a_q025,a_median,a_q975,b_mean,b_q025,b_median,b_q975" and len(rows) == X.shape[1]
    for m, r in enumerate(rows):
        assert int(r[0]) == m
        assert r[1] == "%.6f" % mg["a"]["mean"][m] and [int(v) for v in r[2:5]] == list(mg["a"]["quantiles"][m]), m
        assert r[5] == "%.6f" % mg["b"]["mean"][m] and [int(v) for v in r[6:9]] == list(mg["b"]["quantiles"][m]), m
    # replay-selected: the same marginal files, and po.csv byte-identical to the run without --marginals
    run(["--replay-selected", "--po", str(tmp_path / "p1.csv")])
    out2 = run(["--replay-selected", "--po", str(tmp_path / "p2.csv"), "--marginals", str(tmp_path / "Q")])
    assert (tmp_path / "p2.csv").read_bytes() == (tmp_path / "p1.csv").read_bytes()
    assert pick(out2, "marginals:") == line
    for suffix in (".sites.csv", ".taxa.csv"):
        assert (tmp_path / ("Q" + suffix)).read_bytes() == (tmp_path / ("P" + suffix)).read_bytes()
