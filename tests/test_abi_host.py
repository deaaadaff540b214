"""The C-ABI library: loads, exports every symbol include/seriation_b200.h declares, and its
host-only entry points (readers, synthetic generator, host selection, PO finalisation) behave like
the reference.  No compute calls: this file runs without a GPU."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import NOW, ROOT, load_hex_dataset


@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


def test_every_declared_symbol_is_exported(S):
    header = open(os.path.join(ROOT, "include", "seriation_b200.h")).read()
    declared = set(re.findall(r"\b(ser_[a-z0-9_]+)\s*\(", header))
    declared -= {"ser_run_config"}
    bound = {name for name, _, _ in S.SYMBOLS}
    assert declared == bound, declared ^ bound
    L = S.lib()
    for name in declared:
        assert hasattr(L, name), name
    assert b"sm_100a" in L.ser_version()


@pytest.mark.parametrize("name", NOW)
def test_txt_reader_matches_oracle_parser(S, oracle_mod, tmp_path, name):
    X, hard = load_hex_dataset(name)
    p = tmp_path / (name + ".txt")
    p.write_text(oracle_mod.format_dataset(X, hard))
    ds = S.Dataset.read_txt(str(p))
    X2, h2 = ds.arrays()
    assert (ds.N, ds.M, ds.nh) == (X.shape[0], X.shape[1], int(hard.sum()))
    assert np.array_equal(X, X2) and np.array_equal(hard, h2)
    Xo, ho = oracle_mod.load_dataset(str(p))
    assert np.array_equal(Xo, X2) and np.array_equal(ho, h2)


def test_txt_reader_grammar_quirks(S, tmp_path):
    # any separator, '*' anywhere after the M-th cell, short rows zero-filled (mcmc.c:366-400)
    p = tmp_path / "q.txt"
    p.write_text("3 4\n1,0;1 1 *\n0011 trailing\n1 1\n")
    X, hard = S.Dataset.read_txt(str(p)).arrays()
    assert X.tolist() == [[1, 0, 1, 1], [0, 0, 1, 1], [1, 1, 0, 0]]
    assert hard.tolist() == [1, 0, 0]
    # a '*' between cells is skipped like any separator and does not mark the site
    p.write_text("1 3\n1 * 0 1\n")
    X, hard = S.Dataset.read_txt(str(p)).arrays()
    assert X.tolist() == [[1, 0, 1]] and hard.tolist() == [0]


@pytest.mark.parametrize("text", ["", "x y\n", "0 4\n", "2 2\n1 0\n"])
def test_txt_reader_errors(S, tmp_path, text):
    p = tmp_path / "bad.txt"
    p.write_text(text)
    with pytest.raises(S.SeriationError) as e:
        S.Dataset.read_txt(str(p))
    assert "read error" in str(e.value)  # the reference's own messages (mcmc.c:349,355,371)


def test_genus_and_sites_readers(S, tmp_path):
    X = np.eye(3, 2, dtype=np.uint8)
    ds = S.Dataset.from_bits(X, np.array([0, 1, 0], np.uint8))
    g = tmp_path / "t.genus"
    s = tmp_path / "t.sites"
    g.write_text("Pseudocyon \nHemicyon \n")
    s.write_text("Laugnac [2,21.38] *\nEsvres___Continental_Sands [3,19.5]\nWintershof_West [3,19] *\n")
    ds.read_names(str(g), str(s))
    assert ds.taxon_name(1) == "Hemicyon" and ds.site_name(1) == "Esvres___Continental_Sands"
    assert ds.site_age(0) == (2, 21.38, True) and ds.site_age(1) == (3, 19.5, False)
    g.write_text("only_one\n")
    with pytest.raises(S.SeriationError):
        ds.read_names(str(g), None)


def test_synthetic_generator(S):
    ds = S.Dataset.synthetic(1024, 4096, 16)
    X, hard = ds.arrays()
    assert X.shape == (1024, 4096) and hard.sum() == 16
    assert X.any(axis=0).all() and X.any(axis=1).all()
    assert 0.03 < X.mean() < 0.12
    X2, h2 = S.Dataset.synthetic(1024, 4096, 16).arrays()
    assert np.array_equal(X, X2) and np.array_equal(hard, h2)  # deterministic
    small = S.Dataset.synthetic(40, 25, 3, 7)
    assert small.nh == 3


def test_host_selection_matches_script_semantics(S, oracle_mod):
    rng = np.random.default_rng(3)
    for n, k in ((100, 8), (100, 2), (7, 3), (1, 1), (4096, 2)):
        e = rng.normal(5000, 40, n)
        got, mn, sd = S.select_chains(e, k)
        assert list(got) == oracle_mod.choose_chains(e, k)
        assert mn == e.min() and abs(sd - np.std(e)) <= 1e-12 * max(1.0, np.std(e))
    assert list(S.select_chains(np.array([3.0]), 1)[0]) == []  # one chain: sigma = 0, strict -> empty


def test_po_finalize_matches_script_semantics(S, oracle_mod):
    rng = np.random.default_rng(5)
    N, T = 17, 40
    per_chain = []
    for c in range(3):
        pis = np.array([rng.permutation(N) for _ in range(T)])
        per_chain.append(oracle_mod.pair_order_counts(pis))
    counts = np.stack(per_chain).astype(np.int32)
    for faithful in (True, False):
        want = oracle_mod.pair_order_matrix(per_chain, 3, faithful)
        got = S.po_finalize(counts, 3, faithful)
        assert np.allclose(got, want, rtol=0, atol=1e-15)


def test_posterior_summary_finalisers_match_script_semantics(S, oracle_mod):
    """compute_exp_ages / compute_exp_pi / compute_exp_a (script.py:129-152, :230-276) incl. their
    reset / carry-over quirks, from per-chain sums (the GPU produces the sums)."""
    rng = np.random.default_rng(9)
    N, M, T, k = 19, 11, 30, 3
    pis = [np.array([rng.permutation(N) for _ in range(T)]) for _ in range(k)]
    a_s = [rng.integers(0, N, size=(T, M)) for _ in range(k)]
    corr_num = np.array([int((p * np.arange(N)).sum()) for p in pis])
    r = S.pearson_from_corr_num(corr_num, T, N)
    for c in range(k):
        want = np.mean([np.corrcoef(p, np.arange(N))[0, 1] for p in pis[c]])
        assert abs(r[c] - want) < 1e-12
    assert abs(float(np.sum(r * T / 1000) / k) - oracle_mod.exp_ages(pis, k)) < 1e-12
    got_pi = S.carry_over_mean([p.sum(axis=0) for p in pis], k, keep_total=False)
    assert np.allclose(got_pi, oracle_mod.exp_pi(pis, k), rtol=0, atol=1e-12)
    got_a = S.carry_over_mean([a.sum(axis=0) for a in a_s], k, keep_total=True)
    assert np.allclose(got_a, oracle_mod.exp_a(a_s, k), rtol=0, atol=1e-12)
    clean = S.carry_over_mean([p.sum(axis=0) for p in pis], k, keep_total=False, faithful=False)
    assert np.allclose(clean, sum(p.sum(axis=0) for p in pis) / 1000 / k)


def test_probability_map_finalisers_match_script_semantics(S, oracle_mod):
    """taxa_occurence_ / false_taxa_occurence_ / false_ones_probability_matrix (script.py:306-448) from per-chain
    alive counts: the host finalisers (carry-over, E[pi] / E[a] reordering) against the numpy restatements
    that are pinned to the unmodified script.py.  The device reductions are replaced by numpy here."""
    rng = np.random.default_rng(17)
    N, M, T, k = 23, 13, 40, 3
    X = (rng.random((N, M)) < 0.3).astype(np.uint8)
    pis = [np.array([rng.permutation(N) for _ in range(T)]) for _ in range(k)]
    a_s = [rng.integers(0, N // 2, size=(T, M)) for _ in range(k)]
    b_s = [a + rng.integers(0, N // 2, size=(T, M)) for a in a_s]

    class FakeRun:
        N, M = 23, 13
        ds = S.Dataset.from_bits(X)

        def alive_counts(self, chosen):
            j = np.arange(N)[None, :, None]
            return np.stack([((j >= a_s[c][:, None, :]) & (j <= b_s[c][:, None, :])).sum(axis=0) for c in chosen]).astype(np.int32), T

        def posterior_sums(self, chosen, with_ab=False):
            out = dict(corr_num=np.array([int((pis[c] * np.arange(N)).sum()) for c in chosen]), n_samples=T,
                       pi_sum=np.stack([pis[c].sum(axis=0) for c in chosen]))
            if with_ab:
                out.update(a_sum=np.stack([a_s[c].sum(axis=0) for c in chosen]), b_sum=np.stack([b_s[c].sum(axis=0) for c in chosen]))
            return out

    batch = S.ChainBatch(FakeRun(), 0, T)
    chains = [0, 1, 2]
    assert np.allclose(S.taxa_occurence_probability_matrix(batch, chains, k), oracle_mod.alive_matrix(a_s, b_s, pis, k), rtol=0, atol=1e-13)
    assert np.allclose(S.false_taxa_occurence_probability_matrix(batch, chains, k), oracle_mod.false_taxa_matrix(a_s, b_s, pis, k), rtol=0, atol=1e-13)
    assert np.allclose(S.false_ones_probability_matrix(batch, chains, k), oracle_mod.false_ones_matrix(a_s, b_s, pis, k, X), rtol=0, atol=1e-13)
    Y = S.new_data_matrix(batch, chains, k)
    assert Y.shape == (N, M) and Y.sum() == X.sum()


# ----------------------------------------------------------------------------- the ABI struct and INTEGRATION.md
def _integration_snippet():
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    level2 = text[text.index("## Level 2"):]
    return level2[level2.index("```python\n") + len("```python\n"):level2.index("\n```\n")]


def test_integration_snippet_matches_the_abi(S):
    """INTEGRATION.md's ctypes RunConfig, api.RunConfig and the header's ser_run_config list the same fields in
    the same order with the same widths (round 1 shipped a doc struct one field short)."""
    header = open(os.path.join(ROOT, "include", "seriation_b200.h")).read()
    body = header[header.index("typedef struct ser_run_config {"):header.index("} ser_run_config;")]
    h_fields = re.findall(r"^\s*(u?int32_t)\s+([a-z_]+);", body, re.M)
    ctype = {"int32_t": C.c_int32, "uint32_t": C.c_uint32}
    want = [(name, ctype[t]) for t, name in h_fields]
    assert len(want) == 10 and want[0][0] == "struct_size"
    assert [(n, t) for n, t in S.RunConfig._fields_] == want
    ns = {}
    snippet = _integration_snippet()
    exec(snippet[snippet.index("class RunConfig"):snippet.index("n_chains, burn, samples, k =")], {"C": C}, ns)
    assert [(n, t) for n, t in ns["RunConfig"]._fields_] == want
    assert C.sizeof(ns["RunConfig"]) == C.sizeof(S.RunConfig) == 4 * len(want)


def test_run_create_refuses_a_struct_of_another_size(S):
    """a caller built against another layout is refused before anything is read past its struct"""
    ds = S.Dataset.from_bits(np.eye(4, 3, dtype=np.uint8))
    cfg = S.RunConfig(C.sizeof(S.RunConfig) - 4, 1, 0, 10, 0, 0, 0, 0, 0, 0)
    h = C.c_void_p()
    assert S.lib().ser_run_create(ds._h, C.byref(cfg), C.byref(h)) == -1 and not h.value
    assert b"struct_size" in S.lib().ser_last_error()
    assert S.lib().ser_multi_create(ds._h, C.byref(cfg), 1, None, C.byref(h)) == -1 and not h.value


def test_compute_entry_points_fail_loudly_without_a_device(S):
    """no CPU fallback: on a box without a GPU every compute entry point says so"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    ds = S.Dataset.from_bits(np.eye(4, 3, dtype=np.uint8))
    with pytest.raises(S.SeriationError) as e:
        S.Run(ds, 2)
    assert "no CUDA device" in str(e.value) and "no CPU path" in str(e.value)
    with pytest.raises(S.SeriationError) as e:
        S.Multi(ds, 4, 2)
    assert "no CUDA device" in str(e.value)


def test_warp_batch_plan_of_the_large_shape_kernel(S):
    """ser_plan_warp_batches (host only): the batches cover every sorted column exactly once and in order, a batch's items fit a
    warp's slice, it has at most 32 columns, every column gets a power of two of lanes, the lanes of a batch fit one warp, and a
    batch that would leave more than 4 lanes idle holds a power of two of columns (all 32 lanes busy) unless it is the matrix's tail"""
    rng = np.random.default_rng(3)
    cases = [(np.sort(rng.integers(18, 166, 4096))[::-1], 600),      # the 1024 x 4096 synthetic shape: 19 .. 166 items per column
             (np.sort(rng.integers(0, 40, 1500))[::-1], 200), (np.full(77, 1023), 1024), (np.zeros(500, np.int64), 8),
             (np.sort(rng.integers(0, 2049, 300))[::-1], 4096), (np.array([5]), 16)]
    for ones, wcap in cases:
        plan = S.plan_warp_batches(ones, wcap)
        off = np.concatenate([[0], np.cumsum(ones + 1)])
        nxt = 0
        for c0, nc, lsh, e0, e1 in plan.tolist():
            assert c0 == nxt and 1 <= nc <= 32 and (nc << lsh) <= 32 and (nc << (lsh + 1)) > 32
            assert e0 == off[c0] and e1 == off[c0 + nc] and e1 - e0 <= wcap
            fits = nc                                                 # how many columns would have fitted
            while c0 + fits < ones.size and fits < 32 and off[c0 + fits + 1] - e0 <= wcap:
                fits += 1
            if fits != nc:                                            # shrunk: to the largest power of two, all lanes busy
                assert nc & (nc - 1) == 0 and 2 * nc > fits and (nc << lsh) == 32
            elif (nc << lsh) < 28:                                    # idle lanes are only left at the matrix's tail
                assert c0 + (1 << (nc.bit_length() - 1)) >= ones.size
            nxt = c0 + nc
        assert nxt == ones.size
    with pytest.raises(S.SeriationError):
        S.plan_warp_batches(np.array([100, 3]), 50)                  # a column wider than a slice: the CTA-wide groups serve such shapes
