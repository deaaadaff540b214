"""The cross-chain reductions against plain numpy and the oracle, at the edges of their tiles, chunks and shapes: the chain
selector on constructed vectors (ties across threads and warps, values exactly on the window edge, k beyond the candidates,
up to 524 288 chains); the one-shot pair-order counts, posterior sums and alive counts on real stores (N and M on both sides
of 32, 128 and 256, sample counts on both sides of the 32-sample staging chunk); the streaming accumulators over windows
that do not divide the sample count; and every reduction and histogram over crafted stores injected through a checkpoint,
with a, b and pi at the ends of their ranges."""
import os
import struct

import numpy as np
import pytest

from conftest import load_hex_dataset, random_dataset
from test_checkpoint import _layout, _patch_record


@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


# ----------------------------------------------------------------------------- chain selection on constructed vectors
SMALL_N = (1, 2, 31, 32, 33, 1023, 1024, 1025)
LARGE_N = (65536, 524288)


def _ks(n):
    """k in {1, 2, 8, n}; at the large n, where k rounds of a scan over n values would take minutes, k = 1, 2, 8 and 64"""
    return (1, 2, 8, n) if n <= 2048 else (1, 2, 8, 64)


def _far_from_the_window_edges(e):
    lo, sd = e.min(), np.std(e)
    for edge in (lo - sd, lo + sd):
        assert np.min(np.abs(e - edge)) > 1e-9 * max(abs(edge), 1e-300), "a value lies within rounding distance of min +- sigma"


def _selection_cases():
    """(name, vector, ks, exact): `exact` vectors have a mean and sigma that every summation order computes exactly"""
    rng = np.random.default_rng(20261020)
    cases = []
    for n in SMALL_N + LARGE_N:
        e = rng.uniform(100.0, 200.0, n)
        if n > 1:                                           # one value: sigma is 0 in any order and the window is empty
            _far_from_the_window_edges(e)
        cases.append(("random %d" % n, e, _ks(n), n == 1))
    # ties: one unique minimum at the last id, then equal values at ids i, i+1 (neighbouring lanes), i+32 (another warp) and
    # i+1024 (the same thread of the 1024-thread CTA); k = 2, 3, 4 cut the tie between the k-th and (k+1)-th candidates
    for n, i in ((1056, 5), (2048, 31), (65536, 1000)):
        e = rng.uniform(1.0, 11.0, n)
        e[n - 1] = 0.0
        e[[i, i + 1, i + 32, i + 1024]] = 0.5
        _far_from_the_window_edges(e)
        cases.append(("ties %d at %d" % (n, i), e, (1, 2, 3, 4, 5, 8) + ((n,) if n <= 2048 else ()), False))
    # {0, 0, 1, 1, 1, 3}: mean 1 and sigma 1 exactly, so the 1s lie on min + sigma and are not candidates; every 0 ties
    for n in (6, 36, 1026, 65532, 524286):
        e = rng.permutation(np.tile(np.array([0.0, 0.0, 1.0, 1.0, 1.0, 3.0]), n // 6))
        cases.append(("edges %d" % n, e, _ks(n), True))
    # all equal: sigma = 0 and the open window is empty
    for n in (1, 32, 1025, 65536):
        cases.append(("equal %d" % n, np.full(n, 7.25), _ks(n), True))
    # a few candidates among many far values: k beyond the candidates at the large n too
    for n in (65536, 524288):
        e = rng.uniform(1000.0, 1001.0, n)
        e[rng.choice(n, 5, replace=False)] = [0.0, 0.25, 0.5, 0.75, 1.0]
        _far_from_the_window_edges(e)
        cases.append(("sparse %d" % n, e, (1, 2, 8, 64), False))
    return cases


_CASES = _selection_cases()


def test_host_selection_equals_the_oracle(S, oracle_mod):
    for name, e, ks, exact in _CASES:
        for k in ks:
            want = oracle_mod.choose_chains(e, k)
            ids, mn, sd = S.select_chains(e, k)
            assert ids.tolist() == want, (name, k)
            assert mn == e.min(), (name, k)
            if exact:
                assert sd == np.std(e) and sd in (0.0, 1.0), (name, k)
            else:
                assert abs(sd - np.std(e)) <= 1e-12 * np.std(e), (name, k)
        if name.startswith("edges"):
            assert len(oracle_mod.choose_chains(e, len(e))) == len(e) // 3       # the 0s, none of the 1s
        if name.startswith("equal"):
            assert oracle_mod.choose_chains(e, len(e)) == []


@pytest.mark.gpu
def test_device_selection_equals_the_oracle_and_the_host(S, oracle_mod):
    import torch
    for name, e, ks, exact in _CASES:
        d_e = torch.tensor(e, dtype=torch.float64, device="cuda")
        for k in ks:
            d_ch = torch.full((k,), -7, dtype=torch.int32, device="cuda")
            d_info = torch.full((3,), -7.0, dtype=torch.float64, device="cuda")
            S.select_chains_device(d_e.data_ptr(), len(e), k, d_ch.data_ptr(), d_info.data_ptr())
            torch.cuda.synchronize()
            got, info = d_ch.cpu().numpy(), d_info.cpu().numpy()
            want = oracle_mod.choose_chains(e, k)
            host, hmn, hsd = S.select_chains(e, k)
            assert got.tolist() == want + [-1] * (k - len(want)), (name, k)
            assert host.tolist() == want, (name, k)
            assert info[0] == len(want) and info[1] == e.min() == hmn, (name, k)
            if exact:
                assert info[2] == hsd == np.std(e), (name, k)
            else:
                assert abs(info[2] - np.std(e)) <= 1e-12 * np.std(e), (name, k)


# ----------------------------------------------------------------------------- numpy references over stored samples
def _sums_ref(s):
    pi = s["pi"].astype(np.int64)
    return dict(pi_sum=pi.sum(axis=0), a_sum=s["a"].astype(np.int64).sum(axis=0), b_sum=s["b"].astype(np.int64).sum(axis=0),
                corr_num=int((pi * np.arange(pi.shape[1])).sum()))


def _alive_ref(a, b, N):
    """#{t : a_t(m) <= j <= b_t(m)} for j < N by a difference array: +1 at a, -1 at b + 1"""
    T, M = a.shape
    diff = np.zeros((N + 2, M), np.int64)
    cols = np.tile(np.arange(M), T)
    np.add.at(diff, (a.ravel(), cols), 1)
    np.add.at(diff, (b.ravel() + 1, cols), -1)
    return np.cumsum(diff, axis=0)[:N]


def _hist_ref(x, bins):
    T, items = x.shape
    h = np.zeros((items, bins), np.int64)
    np.add.at(h, (np.tile(np.arange(items), T), x.ravel()), 1)
    return h


def _check_sums(ps, c, ref, what):
    for key in ("pi_sum", "a_sum", "b_sum"):
        assert np.array_equal(ps[key][c], ref[key]), (what, key)
    assert ps["corr_num"][c] == ref["corr_num"], (what, "corr_num")


def _check_one_shot(oracle_mod, run, chosen, samples, T, what):
    """po_counts, posterior_sums and alive_counts of `chosen` (global = local ids; -1 and repeats allowed) against numpy"""
    N = run.N
    po = run.po_counts(chosen)
    ps = run.posterior_sums(chosen, with_ab=True)
    alive, t_alive = run.alive_counts(chosen)
    assert ps["n_samples"] == t_alive == T, what
    for c, g in enumerate(chosen):
        if g < 0:
            assert not po[c].any() and not ps["pi_sum"][c].any() and not ps["a_sum"][c].any() and ps["corr_num"][c] == 0, what
            assert not alive[c].any(), what
            continue
        s = samples[g]
        assert s["pi"].shape[0] == T, what
        assert np.array_equal(po[c], oracle_mod.pair_order_counts(s["pi"])), (what, g, "po")
        _check_sums(ps, c, _sums_ref(s), (what, g))
        assert np.array_equal(alive[c], _alive_ref(s["a"], s["b"], N)), (what, g, "alive")


def _random_ds(S, N, M, density, seed):
    X, hard = random_dataset(np.random.default_rng(seed), N, M, min(3, N - 1), density)
    return S.Dataset.from_bits(X, hard)


ONE_SHOT_SHAPES = [  # (N, M, density); the last two are the big ones
    (2, 3, .5), (31, 7, .3), (32, 127, .15), (33, 128, .15), (64, 129, .1), (255, 40, .05), (256, 9, .05), (257, 9, .05),
    (2048, 8, .005), "g10s10", "synthetic",
]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ONE_SHOT_SHAPES, ids=lambda s: s if isinstance(s, str) else "%dx%d" % s[:2])
def test_one_shot_reductions_equal_numpy(S, oracle_mod, shape):
    if shape == "g10s10":
        ds, n, spc, steps = S.Dataset.from_bits(*load_hex_dataset("g10s10")), 3, 10, (1, 30, 1, 1, 32, 935)
    elif shape == "synthetic":
        ds, n, spc, steps = S.Dataset.synthetic(1024, 4096), 2, 1, (1, 32, 32)
    else:
        N, M, density = shape
        big = N >= 2048
        ds, n, spc, steps = _random_ds(S, N, M, density, N * 1000 + M), 2 if big else 3, 10, (1, 30, 1, 1, 32)
    T_max = sum(steps)
    run = S.Run(ds, n, seed=31, sweeps_per_call=spc, store=S.STORE_FULL, max_samples=T_max).init().advance(2, False)
    chosen = np.array([n - 1, 0, -1, n - 1] + ([1] if n > 2 else []), np.int32)     # unsorted, a repeat and a -1
    T = 0
    for step in steps:
        run.advance(step, True).sync()
        T += step
        samples = {g: run.fetch_samples(g) for g in range(n)}
        _check_one_shot(oracle_mod, run, chosen, samples, T, (shape, T))
    assert run.check() == 0


# ----------------------------------------------------------------------------- streaming accumulators
STREAM_SHAPES = [(33, 128, .15), (257, 9, .05), "g10s10"]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", STREAM_SHAPES, ids=lambda s: s if isinstance(s, str) else "%dx%d" % s[:2])
def test_streaming_reductions_equal_numpy(S, oracle_mod, shape):
    if shape == "g10s10":
        ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    else:
        ds = _random_ds(S, shape[0], shape[1], shape[2], 7 + shape[0])
    N, M, n, burn, T, seed = ds.N, ds.M, 3, 3, 65, 17
    chosen = np.array([2, 0, -1, 2], np.int32)
    ref = S.Run(ds, n, seed=seed, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    samples = {g: ref.fetch_samples(g) for g in range(n)}
    want_po = {g: oracle_mod.pair_order_counts(samples[g]["pi"]) for g in range(n)}
    for W in (1, 7, 32, 33):
        run = S.Run(ds, n, seed=seed, store=S.STORE_FULL, max_samples=W).init()
        run.accumulate(ab=True, alive=True, positions=True, ranges=True)
        run.advance_both(burn, 5).advance(T - 5, True).sync()                 # 5 and 60 samples: neither is a multiple of W
        po = run.po_counts(chosen)
        ps = run.posterior_sums(chosen, with_ab=True)
        alive, t_alive = run.alive_counts(chosen)
        m = run.marginals(chosen, ranges=True)
        assert ps["n_samples"] == t_alive == T and m["n_samples"].tolist() == [T, T, 0, T], W
        for c, g in enumerate(chosen):
            if g < 0:
                assert not po[c].any() and not alive[c].any() and not m["pos"][c].any() and not m["a"][c].any(), W
                continue
            s, what = samples[g], (shape, W, int(g))
            assert np.array_equal(po[c], want_po[g]), what
            _check_sums(ps, c, _sums_ref(s), what)
            assert np.array_equal(alive[c], _alive_ref(s["a"], s["b"], N)), what
            assert np.array_equal(m["pos"][c], _hist_ref(s["pi"], N)), what
            assert np.array_equal(m["a"][c], _hist_ref(s["a"], N + 1)) and np.array_equal(m["b"][c], _hist_ref(s["b"], N + 1)), what
        run.close()


# ----------------------------------------------------------------------------- crafted stores through a checkpoint
def _crafted_pi(rng, N, T, c):
    rows = []
    for t in range(T):
        kind = (t + c) % 4
        if kind == 0:
            rows.append(np.arange(N))
        elif kind == 1:
            rows.append(np.arange(N)[::-1])
        elif kind == 2:
            rows.append(np.roll(np.arange(N), 1))
        else:
            rows.append(rng.permutation(N))
    return np.array(rows, np.uint16)


def _crafted_ab(rng, N, M, T):
    """per taxon and row an (a, b) pair at the ends of the range (a <= b <= N), cycling, with mid-range pairs in between"""
    edges = [(0, 0), (0, N), (N, N), (N - 1, N), (N - 1, N - 1), (0, 1)]
    a, b = np.empty((T, M), np.uint16), np.empty((T, M), np.uint16)
    for t in range(T):
        for m in range(M):
            q = (t * 7 + m) % (len(edges) + 2)
            if q < len(edges):
                a[t, m], b[t, m] = edges[q]
            else:
                lo, hi = np.sort(rng.integers(1, N, 2))
                a[t, m], b[t, m] = lo, hi
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("N,M", [(33, 37), (257, 20)])
def test_crafted_stores_through_a_checkpoint(S, oracle_mod, tmp_path, N, M):
    ds = _random_ds(S, N, M, .1, N + M)
    n, R, kw = 4, 33, dict(seed=5, store=S.STORE_FULL, max_samples=33)
    f = str(tmp_path / "ck")
    saved = S.Run(ds, n, **kw).init().advance(2, False).advance(R, True).save_checkpoint(f).sync()
    data = open(f, "rb").read()
    size = struct.unpack_from("<Q", data, 88)[0]
    L = _layout(N, M, 0, S.STORE_FULL, R, 0)
    assert L["size"] == size and struct.unpack_from("<i", data, 80)[0] == R
    first = 104 + (4 * n + 7) // 8 * 8 + 8
    for c in range(n):                                      # the records' rows are the store's rows, in sample order
        rec, s = data[first + c * size:first + (c + 1) * size], saved.fetch_samples(c)
        for key, off, width in (("pi", L["spi"], N), ("a", L["sa"], M), ("b", L["sb"], M)):
            rows = np.frombuffer(rec, np.uint16, R * width, off).reshape(R, width)
            assert np.array_equal(rows, s[key]), (c, key)
    saved.close()

    rng = np.random.default_rng(N * M)
    own = [1, 31, 32, 33]                                   # the chains' own sample counts
    crafted = {}
    for c in range(n):
        pi = _crafted_pi(rng, N, R, c)
        a, b = _crafted_ab(rng, N, M, R)
        crafted[c] = dict(pi=pi[:own[c]].astype(np.int64), a=a[:own[c]].astype(np.int64), b=b[:own[c]].astype(np.int64))

        def edit(rec, L, pi=pi, a=a, b=b, t=own[c]):
            rec[L["spi"]:L["spi"] + pi.nbytes] = pi.tobytes()
            rec[L["sa"]:L["sa"] + a.nbytes] = a.tobytes()
            rec[L["sb"]:L["sb"] + b.nbytes] = b.tobytes()
            struct.pack_into("<i", rec, 156, t)
        patched = _patch_record(f, c, edit)
        open(f, "wb").write(patched)
    run = S.Run(ds, n, **kw).load_checkpoint(f)
    chosen = [3, 1, 0, 2]
    po = run.po_counts(chosen)
    m = run.marginals(chosen, ranges=True)
    assert m["n_samples"].tolist() == [own[g] for g in chosen]
    for c, g in enumerate(chosen):
        s, T, what = crafted[g], own[g], (N, M, g)
        assert np.array_equal(po[c], oracle_mod.pair_order_counts(s["pi"])), what
        ps = run.posterior_sums([g], with_ab=True)          # one chain per call: it refuses chains whose sample counts differ
        assert ps["n_samples"] == T, what
        _check_sums(ps, 0, _sums_ref(s), what)
        alive, t_alive = run.alive_counts([g])
        assert t_alive == T and np.array_equal(alive[0], _alive_ref(s["a"], s["b"], N)), what
        assert np.array_equal(m["pos"][c], _hist_ref(s["pi"], N)), what
        for key in ("a", "b"):
            h = _hist_ref(s[key], N + 1)
            assert np.array_equal(m[key][c], h) and h[:, N].any(), (what, key)   # bin N is counted
            assert np.all(m[key][c].sum(axis=1) == T), (what, key)
        assert np.all(m["pos"][c].sum(axis=1) == T), what
    assert run.check() == 0
