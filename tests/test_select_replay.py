"""Select-then-replay: runs over an explicit list of global chain ids (ser_run_create_chains) and summaries that accumulate
through a windowed sample store (ser_run_accumulate), checked against the one-shot path that stores every sample."""
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


# ----------------------------------------------------------------------------- host-only argument checks
def test_create_chains_checks_its_arguments_before_any_cuda_call(S):
    ds = S.Dataset.from_bits(np.eye(6, 4, dtype=np.uint8))
    assert "listed twice" in _raises(S, E_ARG, S.Run, ds, 0, chain_ids=[4, 2, 4])
    assert "negative" in _raises(S, E_ARG, S.Run, ds, 0, chain_ids=[3, -1])
    assert "chain_offset" in _raises(S, E_ARG, S.Run, ds, 0, chain_offset=5, chain_ids=[0, 1])
    ids = np.array([1, 2, 3], np.int32)
    cfg = S.RunConfig(C.sizeof(S.RunConfig), 2, 0, 10, S.MODE_FREE, 0, S.STORE_PI, 4, 0, 0)
    h = C.c_void_p()
    assert S.lib().ser_run_create_chains(ds._h, C.byref(cfg), ids.ctypes.data_as(C.POINTER(C.c_int32)), 3, C.byref(h)) == E_ARG
    assert not h.value and b"n_chains = 2" in S.lib().ser_last_error()


def test_accumulate_without_a_run(S):
    assert S.lib().ser_run_accumulate(None, S.ACC_PO) == E_ARG


# ----------------------------------------------------------------------------- GPU
def _same_state(x, y, what):
    assert x.keys() == y.keys()
    for k in x:
        assert np.array_equal(x[k], y[k]), (what, k)


PATHS = {"default": {}, "big_groups": {"SER_FORCE_BIG": "256", "SER_BIG_WARP": "0"},
         "big_warp": {"SER_FORCE_BIG": "256", "SER_BIG_WARP": "1"}, "manycd": {}}


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", [("g10s10", p) for p in PATHS] + [("g2s2", "default")])
def test_subset_run_is_bit_identical_to_the_first_run(S, monkeypatch, tmp_path, name, path):
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)
    ds = S.Dataset.from_bits(*load_hex_dataset(name))
    ids, burn, samp, many = [31, 2, 17], 6, 5, path == "manycd"
    full = S.Run(ds, 40, seed=11, store=S.STORE_FULL, max_samples=samp, manycd=many).init()
    sub = S.Run(ds, 0, seed=11, store=S.STORE_FULL, max_samples=samp, manycd=many, chain_ids=ids).init()
    assert sub.n_chains == 3 and sub.kernel_path() == full.kernel_path()
    for c, g in enumerate(ids):
        _same_state(sub.state(c), full.state(g), ("init", g))
    full.advance(burn, False).advance(samp, True).sync()
    sub.advance(burn, False).advance(samp, True).sync()
    fs, ss = full.chain_stats(), sub.chain_stats()
    assert ss["n_samples"] == fs["n_samples"] == samp
    for c, g in enumerate(ids):
        _same_state(sub.state(c), full.state(g), ("final", g))
        assert np.array_equal(sub.counters(c), full.counters(g))
        for k in ("e_negloglik", "e_c", "e_d"):
            assert ss[k][c] == fs[k][g], (g, k)
        _same_state(sub.fetch_samples(c), full.fetch_samples(g), ("samples", g))
        if many:
            assert np.array_equal(np.stack(sub.cd(c)), np.stack(full.cd(g)))
    assert sub.check() == 0
    if path == "default" and name == "g10s10":
        (tmp_path / "a").mkdir()
        (tmp_path / "b").mkdir()
        sub.write_chain_files(1, str(tmp_path / "a"))
        full.write_chain_files(2, str(tmp_path / "b"))
        files = sorted(os.listdir(tmp_path / "b"))
        assert sorted(os.listdir(tmp_path / "a")) == files and len(files) == 5
        for f in files:
            assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f


def _dataset_with_ages(S, tmp_path):
    X, hard = load_hex_dataset("g10s10")
    N, M = X.shape
    rng = np.random.default_rng(5)
    mn = np.sort(rng.integers(2, 14, N))
    age = np.round(22.0 - 1.1 * mn + rng.random(N) * 0.5, 2)
    (tmp_path / "t.genus").write_text("".join("G%d \n" % m for m in range(M)))
    (tmp_path / "t.sites").write_text("".join("S%d [%d,%s]%s\n" % (n, mn[n], repr(float(age[n])), " *" if hard[n] else "") for n in range(N)))
    return S.Dataset.from_bits(X, hard).read_names(str(tmp_path / "t.genus"), str(tmp_path / "t.sites"))


def _summaries(run, chosen):
    ps = run.posterior_sums(chosen, with_ab=True)
    alive, t_alive = run.alive_counts(chosen)
    return dict(po=run.po_counts(chosen), corr=ps["corr_num"], pi=ps["pi_sum"], a=ps["a_sum"], b=ps["b_sum"], t=ps["n_samples"],
                alive=alive, t_alive=t_alive, age=run.site_age_corr(chosen))


def _same_summaries(x, y, what):
    for k in x:
        assert np.array_equal(np.asarray(x[k]), np.asarray(y[k])), (what, k)


@pytest.mark.gpu
def test_streaming_summaries_equal_the_one_shot_store(S, tmp_path):
    ds = _dataset_with_ages(S, tmp_path)
    burn, T, chosen = 5, 50, np.array([1, 4, 99], np.int32)   # 99: held by no run here, its slab stays untouched
    ref = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=T).init().advance(burn, False).advance(T, True).sync()
    want = _summaries(ref, chosen)
    assert want["t"] == T and np.all(want["po"][2] == 0) and np.all(want["pi"][2] == 0)
    for W in (1, 5, 16, 50, 64):
        whole = S.Run(ds, 6, seed=4, store=S.STORE_FULL, max_samples=W).init().accumulate(ab=True, alive=True)
        whole.advance(burn, False).advance(T, True).sync()
        _same_summaries(_summaries(whole, chosen), want, ("contiguous", W))
        sub = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=W, chain_ids=[4, 1]).init().accumulate(ab=True, alive=True)
        sub.advance(burn, False).advance(T, True).sync()
        _same_summaries(_summaries(sub, chosen), want, ("subset", W))
    # sampling calls split over advances that do not line up with the window, burn-in in the same launch as the first ones
    odd = S.Run(ds, 0, seed=4, store=S.STORE_FULL, max_samples=16, chain_ids=[1, 4]).init().accumulate(ab=True, alive=True)
    odd.advance_both(burn, 7).advance(20, True).advance(23, True).sync()
    _same_summaries(_summaries(odd, chosen), want, "split")


@pytest.mark.gpu
def test_a_chosen_id_the_run_does_not_hold_leaves_its_slab_untouched(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    kw = dict(seed=2, store=S.STORE_FULL, chain_ids=[7, 30])
    streaming = S.Run(ds, 0, max_samples=3, **kw).init().accumulate(ab=True, alive=True, positions=True, ranges=True)
    one_shot = S.Run(ds, 0, max_samples=5, **kw).init()
    chosen = np.array([30, 8, 7], np.int32)
    k, N, M = 3, ds.N, ds.M
    i32 = C.POINTER(C.c_int32)
    for what, run in (("streaming", streaming), ("one-shot", one_shot)):
        run.advance(2, False).advance(5, True).sync()
        corr, pi = np.full(k, 7, np.int64), np.full((k, N), 7, np.int32)
        alive, n = np.full((k, N, M), 7, np.int32), C.c_int32()
        po, pos, nm = np.full((k, N, N), 7, np.int32), np.full((k, N, N), 7, np.int32), np.full(k, 7, np.int32)
        ah, bh = np.full((k, M, N + 1), 7, np.int32), np.full((k, M, N + 1), 7, np.int32)
        assert S.lib().ser_run_posterior_sums(run._h, chosen.ctypes.data_as(i32), k, corr.ctypes.data_as(C.POINTER(C.c_int64)),
                                              pi.ctypes.data_as(i32), None, None, C.byref(n)) == 0
        assert S.lib().ser_run_alive_counts(run._h, chosen.ctypes.data_as(i32), k, alive.ctypes.data_as(i32), C.byref(n)) == 0
        assert S.lib().ser_run_po_counts(run._h, chosen.ctypes.data_as(i32), k, po.ctypes.data_as(i32)) == 0
        assert S.lib().ser_run_marginals(run._h, chosen.ctypes.data_as(i32), k, pos.ctypes.data_as(i32), ah.ctypes.data_as(i32),
                                         bh.ctypes.data_as(i32), nm.ctypes.data_as(i32)) == 0
        assert n.value == 5 and corr[1] == 7 and np.all(pi[1] == 7) and np.all(alive[1] == 7), what
        assert np.all(po[1] == 7) and np.all(pos[1] == 7) and np.all(ah[1] == 7) and np.all(bh[1] == 7) and nm.tolist() == [5, 0, 5], what
        assert np.all(pi[[0, 2]].sum(axis=1) == 5 * N * (N - 1) // 2) and np.all(alive[[0, 2]] != 7), what
        # a held slab is written in full, whatever the caller preset: corr_num included
        assert np.array_equal(corr[[0, 2]], pi[[0, 2]].astype(np.int64) @ np.arange(N)), what
        for c, g in ((0, 30), (2, 7)):
            m = run.marginals([g], ranges=True)
            assert np.array_equal(po[c], run.po_counts([g])[0]) and np.all(np.diagonal(po[c]) == -5), (what, g)
            assert np.array_equal(pos[c], m["pos"][0]) and np.array_equal(ah[c], m["a"][0]) and np.array_equal(bh[c], m["b"][0]), (what, g)
    for c, local in ((0, 1), (2, 0)):
        rows = one_shot.fetch_samples(local)["pi"].astype(np.int64)
        assert corr[c] == (rows @ np.arange(N)).sum()


@pytest.mark.gpu
def test_beyond_the_old_store_capacity(S):
    ds = S.Dataset.synthetic(1024, 4096, 16)
    seed, burn, T = 20060206, 2, 40
    sub = S.Run(ds, 0, seed=seed, store=S.STORE_PI, max_samples=8, chain_ids=[3, 40000]).init().accumulate()
    sub.advance(burn, False).advance(T, True).sync()
    for g in (3, 40000):
        one = S.Run(ds, 1, seed=seed, chain_offset=g, store=S.STORE_PI, max_samples=T).init().advance(burn, False).advance(T, True).sync()
        assert np.array_equal(sub.po_counts([g]), one.po_counts([g])), g
        a, b = sub.posterior_sums([g]), one.posterior_sums([g])
        assert a["n_samples"] == b["n_samples"] == T and np.array_equal(a["pi_sum"], b["pi_sum"]) and np.array_equal(a["corr_num"], b["corr_num"])
        one.close()
    # a window of 4 over 1000 samples: every summary counts all of them
    ds10 = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    run = S.Run(ds10, 3, seed=1, store=S.STORE_FULL, max_samples=4).init().accumulate(ab=True, alive=True).advance(1000, True).sync()
    N = ds10.N
    po = run.po_counts([0, 2])
    assert np.all(np.diagonal(po, axis1=1, axis2=2) == -1000)
    off = po + np.transpose(po, (0, 2, 1))
    assert np.all(off[:, ~np.eye(N, dtype=bool)] == 1000)                    # pi_t(i) < pi_t(j) or the reverse, in every sample
    ps = run.posterior_sums([0, 2], with_ab=True)
    assert ps["n_samples"] == 1000 and np.all(ps["pi_sum"].sum(axis=1) == 1000 * N * (N - 1) // 2)
    alive, t = run.alive_counts([0, 2])
    assert t == 1000 and alive.max() <= 1000 and alive.min() >= 0


@pytest.mark.gpu
def test_two_phase_python_flow_equals_the_one_shot_flow(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, burn, samp, k = 64, 20, 30, 3
    one = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_FULL)
    first = S.run_all_chains(ds, n, burn, samp, seed=13, store=S.STORE_NONE)
    chosen = S.choose_chains(first, k)
    assert chosen == S.choose_chains(one, k) and len(chosen) == k
    two = S.replay_chosen(first, chosen, window=16, with_ab=True)
    assert two.run.n_chains == k and two.stats() is first.stats()
    assert np.array_equal(S.compute_pair_order_matrix(two, chosen, k), S.compute_pair_order_matrix(one, chosen, k))
    assert S.compute_exp_ages(two, chosen, k) == S.compute_exp_ages(one, chosen, k)
    assert np.array_equal(S.compute_exp_pi(two, chosen, None, k), S.compute_exp_pi(one, chosen, None, k))
    assert np.array_equal(S.compute_exp_a(two, chosen, k), S.compute_exp_a(one, chosen, k))
    assert S.compute_exp_cd(two, chosen, k) == S.compute_exp_cd(one, chosen, k)
    assert np.array_equal(S.taxa_occurence_probability_matrix(two, chosen, k), S.taxa_occurence_probability_matrix(one, chosen, k))
    # the self-check: a batch whose recorded seed does not produce its chains is refused
    first.seed = 14
    with pytest.raises(S.SeriationError, match="do not reproduce"):
        S.replay_chosen(first, chosen)


@pytest.mark.gpu
def test_cli_replay_selected_equals_the_one_shot_step(S, tmp_path):
    from tools.datasets import write_txt
    write_txt(str(tmp_path / "g10s10.txt"), *load_hex_dataset("g10s10"))
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "200", "--burn", "20", "--samples", "30", "--select", "3",
            "--dataset", str(tmp_path / "g10s10.txt")]
    a = subprocess.run(base + ["--po", str(tmp_path / "A.csv")], check=True, capture_output=True, text=True).stdout.splitlines()
    b = subprocess.run(base + ["--replay-selected", "--window", "7", "--po", str(tmp_path / "B.csv")], check=True, capture_output=True,
                       text=True).stdout.splitlines()
    pick = lambda lines, head: [x for x in lines if x.startswith(head)]
    assert len(pick(a, "selection:")) == 1 and pick(a, "selection:") == pick(b, "selection:")
    assert len(pick(a, "E[c]")) == 1 and pick(a, "E[c]") == pick(b, "E[c]")
    assert (tmp_path / "A.csv").read_bytes() == (tmp_path / "B.csv").read_bytes()


@pytest.mark.gpu
def test_accumulator_error_paths(S):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    run = S.Run(ds, 2, seed=1, store=S.STORE_FULL, max_samples=4).init().advance(1, True)
    assert "already taken samples" in _raises(S, E_STATE, run.accumulate)
    _raises(S, E_STATE, S.Run(ds, 2, store=S.STORE_NONE, max_samples=4).init().accumulate)
    pi_only = S.Run(ds, 2, store=S.STORE_PI, max_samples=4).init()
    assert "SER_STORE_FULL" in _raises(S, E_STATE, pi_only.accumulate, ab=True)
    assert "SER_STORE_FULL" in _raises(S, E_STATE, pi_only.accumulate, po=False, alive=True)
    _raises(S, E_ARG, S.Run(ds, 2, store=S.STORE_PI, max_samples=0).init().accumulate)
    acc = S.Run(ds, 2, store=S.STORE_FULL, max_samples=4).init().accumulate()
    _raises(S, E_STATE, acc.accumulate)
    acc.advance(6, True).sync()
    assert "transient window" in _raises(S, E_STATE, acc.fetch_samples, 0)
    _raises(S, E_STATE, acc.alive_counts, [0])                       # not accumulated
    _raises(S, E_STATE, acc.posterior_sums, [0], with_ab=True)
    _raises(S, E_STATE, acc.cross_chain, 1)
    assert acc.posterior_sums([0])["n_samples"] == 6
