"""Convergence diagnostics over the stored samples: per-chain mean, variance, halves and Geyer ESS on the device
(ser_run_diagnostics), split-R-hat on the host (ser_split_rhat), checked against a NumPy float64 reference."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import load_hex_dataset

E_ARG, E_STATE = -1, -4


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


# ----------------------------------------------------------------------------- NumPy reference (DESIGN.md 3.7)
def ref_stats(x, max_lag=0):
    """mean, var, ess, lags, (mean1, var1, mean2, var2) of one trace"""
    x = np.asarray(x, np.float64)
    T, n = x.size, x.size // 2
    h1, h2 = x[:n], x[T - n:]
    half = lambda h: (h[0], 0.0) if h.min() == h.max() else (h.mean(), h.var(ddof=1))   # a constant half: exactly its value, 0
    halves = (*half(h1), *half(h2))
    if x.min() == x.max():
        return x[0], 0.0, np.nan, 0, (x[0], 0.0, x[0], 0.0)
    y = x - x.mean()
    g0 = np.dot(y, y) / T
    L = min(T, max_lag) if max_lag > 0 else T
    psum, prev, lags, m = 0.0, np.inf, 0, 0
    while 2 * m + 1 < L:
        P = (np.dot(y[:T - 2 * m], y[2 * m:]) / T) / g0 + (np.dot(y[:T - 2 * m - 1], y[2 * m + 1:]) / T) / g0
        if not P > 0:
            break
        P = min(P, prev)
        prev, psum, lags, m = P, psum + P, lags + 2, m + 1
    tau = max(-1.0 + 2.0 * psum, 1.0 / np.log10(T))
    return x.mean(), x.var(ddof=1), T / tau, lags, halves


def ref_rhat(halves, n):
    """BDA3 11.4 over the 2k half-sequences: halves [k][Q][4]"""
    means = np.concatenate([halves[:, :, 0], halves[:, :, 2]])
    var = np.concatenate([halves[:, :, 1], halves[:, :, 3]])
    W = var.mean(axis=0)
    B_n = means.var(axis=0, ddof=1)
    with np.errstate(invalid="ignore", divide="ignore"):
        return np.where(W > 0, np.sqrt(((n - 1) / n * W + B_n) / W), np.nan)


def traces(run, chain):
    s = run.fetch_samples(chain)
    return np.column_stack([-s["loglik"], np.exp(s["c"]), np.exp(s["d"]), s["pi"].astype(np.float64)])


def ar1(phi, T, seed):
    rng = np.random.default_rng(seed)
    e = rng.standard_normal(T)
    x = np.empty(T)
    x[0] = e[0] / np.sqrt(1 - phi * phi)
    for t in range(1, T):
        x[t] = phi * x[t - 1] + e[t]
    return x


# ----------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("phi", [0.0, 0.5, 0.9])
def test_reference_ess_on_ar1(phi):
    x = ar1(phi, 100_000, seed=int(phi * 10) + 1)
    _, _, ess, lags, _ = ref_stats(x)
    tau = x.size / ess
    assert abs(tau / ((1 + phi) / (1 - phi)) - 1) < 0.05, (phi, tau, lags)


def test_reference_ess_floor_on_an_alternating_trace():
    T = 1000
    x = np.tile([0.0, 1.0], T // 2)
    _, _, ess, lags, _ = ref_stats(x)
    assert ess == T / (1 / np.log10(T)) and lags == T


@pytest.mark.parametrize("k", [1, 2, 7])
def test_split_rhat_matches_bda3(S, k):
    rng = np.random.default_rng(k)
    Q, T = 11, 101
    halves = np.empty((k, Q, 4))
    halves[:, :, [0, 2]] = rng.normal(3.0, 0.5, (k, Q, 2))
    halves[:, :, [1, 3]] = rng.gamma(2.0, 1.0, (k, Q, 2))
    got = S.split_rhat(halves, np.full(k, T, np.int32))
    want = ref_rhat(halves, T // 2)
    assert np.all(np.abs(got / want - 1) < 1e-12)


def test_split_rhat_nan_and_refusals(S):
    halves = np.ones((2, 3, 4))
    halves[:, 1, [1, 3]] = 0.0       # W = 0
    halves[0, 2, 0] = 5.0            # W = 0 with different means
    halves[:, 2, [1, 3]] = 0.0
    r = S.split_rhat(halves, [10, 10])
    assert np.isfinite(r[0]) and np.isnan(r[1]) and np.isnan(r[2])
    assert "different numbers of samples" in _raises(S, E_ARG, S.split_rhat, halves, [10, 12])
    _raises(S, E_ARG, S.split_rhat, halves, [3, 3])


def test_diagnostics_argument_checks(S):
    L = S.lib()
    chosen, stats, halves, n = np.zeros(1, np.int32), np.zeros(16), np.zeros(16), np.zeros(1, np.int32)
    i32, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    args = lambda: (chosen.ctypes.data_as(i32),)
    for k, what, lag in ((1, 3, 0), (0, 3, 0), (1, 0, 0), (1, 4, 0), (1, 3, -1)):
        assert L.ser_run_diagnostics(None, *args(), k, what, lag, stats.ctypes.data_as(dp), halves.ctypes.data_as(dp),
                                     n.ctypes.data_as(i32)) == E_ARG
        assert b"k = %d, what = %d, max_lag = %d" % (k, what, lag) in L.ser_last_error()


def test_cli_diagnostics_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--diagnostics", str(tmp_path / "d.csv")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "usage" in r.stderr and not (tmp_path / "d.csv").exists()


# ----------------------------------------------------------------------------- GPU
def _check_against_reference(S, run, chosen, max_lag=0):
    dg = run.diagnostics(chosen, max_lag=max_lag)
    k, Q = len(chosen), 3 + run.N
    for c, g in enumerate(chosen):
        X = traces(run, g)
        assert dg["n_samples"][c] == X.shape[0]
        for q in range(Q):
            mean, var, ess, lags, halves = ref_stats(X[:, q], max_lag)
            got = (dg["mean"][c, q], dg["var"][c, q], *dg["halves"][c, q])
            want = (mean, var, *halves)
            assert np.allclose(got, want, rtol=1e-12, atol=0), (g, q, got, want)
            assert dg["lags"][c, q] == lags, (g, q)
            if np.isnan(ess):
                assert np.isnan(dg["ess"][c, q]), (g, q)
            else:
                assert abs(dg["ess"][c, q] / ess - 1) < 1e-9, (g, q, dg["ess"][c, q], ess)
    want_r = ref_rhat(dg["halves"], dg["n_samples"][0] // 2)
    assert np.allclose(dg["rhat"], want_r, rtol=1e-12, atol=0, equal_nan=True)
    n_ref = np.stack([[ref_stats(X[:, q])[4] for q in range(Q)] for X in (traces(run, g) for g in chosen)])
    assert np.allclose(dg["rhat"], ref_rhat(n_ref, dg["n_samples"][0] // 2), rtol=1e-9, atol=0, equal_nan=True)
    return dg


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["g10s10", "g2s2", "synthetic"])
def test_stats_equal_the_reference(S, name):
    if name == "synthetic":
        ds, n, burn, T, spc, chosen = S.Dataset.synthetic(1024, 4096, 16), 3, 2, 40, 1, [2, 0]
    else:
        ds, n, burn, T, spc, chosen = S.Dataset.from_bits(*load_hex_dataset(name)), 8, 30, 301, 10, [5, 1, 6]
    run = S.Run(ds, n, seed=9, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    if name == "g2s2":
        assert run.kernel_path() == 0
    dg = _check_against_reference(S, run, chosen)
    assert np.all(dg["n_samples"] == T)
    # every sample stored: q = 0's mean is the exp_data E[-logL]
    e = run.chain_stats()["e_negloglik"][chosen]
    assert np.all(np.abs(dg["mean"][:, 0] / e - 1) < 1e-13)


@pytest.mark.gpu
def test_a_trace_longer_than_any_staging_buffer(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    run = S.Run(ds, 2, seed=3, sweeps_per_call=1, store=S.STORE_FULL, max_samples=4096).init().advance(4096, True).sync()
    dg = _check_against_reference(S, run, [1, 0])
    assert np.nanmax(dg["lags"]) > 32                    # more than one lag block somewhere


@pytest.mark.gpu
def test_max_lag(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    run = S.Run(ds, 2, seed=3, sweeps_per_call=1, store=S.STORE_FULL, max_samples=600).init().advance(600, True).sync()
    free = run.diagnostics([0, 1])
    for cap in (1, 2, 7, 32, 33, 40, 64, 65):
        capped = _check_against_reference(S, run, [0, 1], max_lag=cap)
        assert np.nanmax(capped["lags"]) <= cap
        same = free["lags"] < cap
        for key in ("ess", "lags"):
            assert np.array_equal(capped[key][same], free[key][same], equal_nan=True), (cap, key)


def _same(x, y, what):
    for key in ("mean", "var", "ess", "lags", "halves", "n_samples"):
        assert np.asarray(x[key]).tobytes() == np.asarray(y[key]).tobytes(), (what, key)


@pytest.mark.gpu
def test_results_do_not_depend_on_the_run_or_the_grid(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    seed, burn, T, chosen = 21, 10, 80, [6, 1, 3]
    kw = dict(seed=seed, store=S.STORE_FULL, max_samples=T)
    full = S.Run(ds, 8, **kw).init().advance(burn, False).advance(T, True).sync()
    want = full.diagnostics(chosen)
    _same(full.diagnostics([3]), {k: (v[2:] if k != "rhat" else v) for k, v in want.items()}, "k = 1")
    sub = S.Run(ds, 0, chain_ids=[3, 6, 1], **kw).init().advance(burn, False).advance(T, True).sync()
    _same(sub.diagnostics(chosen), want, "subset")
    lo = S.Run(ds, 4, **kw).init().advance(burn, False).advance(T, True).sync()
    hi = S.Run(ds, 4, chain_offset=4, **kw).init().advance(burn, False).advance(T, True).sync()
    a, b = lo.diagnostics(chosen), hi.diagnostics(chosen)
    merged = {k: np.where(np.isnan(a[k]), b[k], a[k]) for k in ("mean", "var", "ess", "lags", "halves")}
    merged["n_samples"] = np.maximum(a["n_samples"], b["n_samples"])
    _same(merged, want, "split by chain_offset")
    assert np.array_equal(S.split_rhat(merged["halves"], merged["n_samples"]), want["rhat"], equal_nan=True)
    # stopped mid-sampling, saved, resumed in another run
    part = S.Run(ds, 8, **kw).init().advance(burn, False).advance(T // 2, True).sync()
    part.save_checkpoint(str(tmp_path / "c.ckpt"))
    resumed = S.Run(ds, 8, **kw).load_checkpoint(str(tmp_path / "c.ckpt")).advance(T - T // 2, True).sync()
    _same(resumed.diagnostics(chosen), want, "resumed")


@pytest.mark.gpu
def test_refusals_and_untouched_slabs(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_NONE, max_samples=8).init().advance(8, True).diagnostics, [0], scalars=False)
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=8).init().advance(8, True).sync()
    assert "SER_STORE_FULL" in _raises(S, E_STATE, pi_only.diagnostics, [0])
    d = pi_only.diagnostics([0, 1], scalars=False)
    assert np.all(np.isnan(d["mean"][:, :3])) and not np.any(np.isnan(d["mean"][:, 3:]))
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate().advance(8, True)
    assert "accumulating" in _raises(S, E_STATE, acc.diagnostics, [0])
    assert "not initialised" in _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_FULL, max_samples=8).diagnostics, [0])
    short = S.Run(ds, 2, store=S.STORE_FULL, max_samples=8).init().advance(3, True)
    assert "3 stored samples" in _raises(S, E_STATE, short.diagnostics, [1])
    run = S.Run(ds, 0, seed=2, store=S.STORE_FULL, max_samples=20, chain_ids=[7, 30]).init().advance(20, True).sync()
    for bad in (dict(max_lag=-1), dict(scalars=False, sites=False)):
        _raises(S, E_ARG, run.diagnostics, [7], **bad)
    d = run.diagnostics([30, -1, 8, 7])
    for c in (1, 2):
        assert np.all(np.isnan(d["mean"][c])) and np.all(np.isnan(d["halves"][c])) and d["n_samples"][c] == 0
    assert np.all(d["n_samples"][[0, 3]] == 20) and d["rhat"] is not None and not np.any(np.isnan(d["mean"][[0, 3]]))


def _cli_rows(path):
    lines = open(path).read().splitlines()
    assert lines[0] == "quantity,mean,rhat,ess_min,ess_sum"
    return [ln.split(",")[0] for ln in lines[1:]], np.array([[float(v) for v in ln.split(",")[1:]] for ln in lines[1:]])


@pytest.mark.gpu
def test_cli_diagnostics(S, tmp_path):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp = 20, 60
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "4",
            "--dataset", str(tmp_path / "g10s10.txt")]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env).stdout.splitlines()
    out = run(["--diagnostics", str(tmp_path / "d.csv")])
    line = [x for x in out if x.startswith("diagnostics:")]
    assert len(line) == 1 and "R-hat -logL" in line[0] and "constant" in line[0]
    assert not [x for x in run([]) if x.startswith("diagnostics:")]
    names, rows = _cli_rows(tmp_path / "d.csv")
    N = X.shape[0]
    assert names == ["-logL", "c", "d"] + ["site_%d" % i for i in range(N)]
    # the same chains in Python
    batch = S.run_all_chains(S.Dataset.from_bits(X, hard), 64, burn, samp, seed=0, store=S.STORE_FULL)
    chosen = S.choose_chains(batch, 4)
    assert ("chosen " + " ".join(map(str, chosen))) in [x for x in out if x.startswith("selection:")][0]
    dg = S.diagnostics(batch, chosen)
    with np.errstate(invalid="ignore"), __import__("warnings").catch_warnings():
        __import__("warnings").simplefilter("ignore", RuntimeWarning)
        want = np.column_stack([dg["mean"].mean(axis=0), dg["rhat"], np.nanmin(dg["ess"], axis=0),
                                np.where(np.all(np.isnan(dg["ess"]), axis=0), np.nan, np.nansum(dg["ess"], axis=0))])
    assert np.allclose(rows, want, rtol=1e-14, atol=0, equal_nan=True)
    # replay mode: the same file, and the pair-order matrix of the windowed path
    run(["--replay-selected", "--po", str(tmp_path / "p1.csv")])
    run(["--replay-selected", "--po", str(tmp_path / "p2.csv"), "--diagnostics", str(tmp_path / "d2.csv")])
    assert (tmp_path / "d2.csv").read_bytes() == (tmp_path / "d.csv").read_bytes()
    assert (tmp_path / "p2.csv").read_bytes() == (tmp_path / "p1.csv").read_bytes()


@pytest.mark.gpu
def test_replay_chosen_keeping_every_sample(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    one = S.run_all_chains(ds, 32, 10, 40, seed=5, store=S.STORE_FULL)
    first = S.run_all_chains(ds, 32, 10, 40, seed=5, store=S.STORE_NONE)
    chosen = S.choose_chains(first, 3)
    two = S.replay_chosen(first, chosen, window=0)
    assert two.run.cfg.store == S.STORE_FULL and two.run.cfg.max_samples == 40
    _same(S.diagnostics(two, chosen), S.diagnostics(one, chosen), "replay_chosen(window=0)")
    assert np.array_equal(S.compute_pair_order_matrix(two, chosen, 3), S.compute_pair_order_matrix(one, chosen, 3))
    assert np.array_equal(S.compute_exp_a(two, chosen, 3), S.compute_exp_a(one, chosen, 3))
