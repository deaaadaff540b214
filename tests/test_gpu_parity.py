"""Parity of the CUDA sweep (through the C ABI) with the oracle.  Run on the B200 box.

Replay mode (north_star check 1+2): with the same draw tape, a, b, pi, every integer count and the
tape cursor are bit-identical to the oracle after every thinned sample; c and d carry the tape's own
libm bits; log-likelihood within 1e-9 relative.
Free-running mode: the structured Philox stream is reproduced by the oracle (detmath mode), so the
same comparison holds without a tape.
"""
import os

import numpy as np
import pytest

from conftest import EDGE_SHAPES, GOLDEN, NOW, load_hex_dataset, random_dataset

pytestmark = pytest.mark.gpu
LL_RTOL = 1e-9  # north_star: "per-state log-likelihood agrees within 1e-9 relative in fp64"


@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    S.lib()
    return S


def _oracle_chain(O, X, hard, seed, burn, samp, philox=None, detmath=False):
    o = O.Oracle(X, hard)
    if philox is not None:
        o.source_philox(*philox)
    else:
        o.source_mt(seed)
    o.record(True).detmath(detmath)
    o.randomize()
    init = o.state()
    res = o.run(burn, samp)
    return o, init, res, o.state(), o.tape()


def _cmp_state(got, want, what):
    for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
        assert np.array_equal(got[k], getattr(want, k)), (what, k)
    assert got["slots"] == want.slots, what
    assert got["c"] == want.c and got["d"] == want.d, what
    assert abs(got["loglik"] - want.loglik) <= LL_RTOL * abs(want.loglik), what


def _cmp_samples(got, res, what):
    for k in ("a", "b", "pi"):
        assert np.array_equal(got[k], res[k]), (what, k)
    assert np.array_equal(got["c"], res["c"]) and np.array_equal(got["d"], res["d"]), what
    # every SAVED log-likelihood carries the reference's bits: on sampled sweeps the kernel forms it
    # with the reference's own sequential per-taxon sums (mcmc.c:625-648 and :1214/1435/1630)
    assert np.array_equal(got["loglik"], res["loglik"]), (what, np.max(np.abs(got["loglik"] - res["loglik"])))


def _replay_case(S, O, X, hard, seeds, burn, samp):
    ds = S.Dataset.from_bits(X, hard)
    chains = [_oracle_chain(O, X, hard, s, burn, samp) for s in seeds]
    run = S.Run(ds, len(seeds), mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=samp)
    run.set_tapes([c[4] for c in chains]).init().sync()
    for i, c in enumerate(chains):
        _cmp_state(run.state(i), c[1], ("init", i))
    run.advance(burn, False).advance(samp, True).sync()
    assert run.check() == 0
    stats = run.chain_stats()
    for i, (o, init, res, final, tape) in enumerate(chains):
        _cmp_state(run.state(i), final, ("final", i))
        assert run.state(i)["slots"] == tape.size and run.state(i)["loglik"] == final.loglik
        _cmp_samples(run.fetch_samples(i), res, ("samples", i))
        assert stats["e_negloglik"][i] == res["sums"][0] / samp   # compute_exp_data's running sum, bit for bit
        assert abs(stats["e_c"][i] - res["sums"][1] / samp) <= 1e-12
        assert abs(stats["e_d"][i] - res["sums"][2] / samp) <= 1e-12
    run.close()


@pytest.mark.parametrize("name,burn,samp", [("g10s10", 20, 20), ("g10s2", 4, 4), ("g5s5", 5, 5), ("g2s2", 4, 4)])
def test_replay_bit_exact_now_subsets(S, oracle_mod, name, burn, samp):
    X, hard = load_hex_dataset(name)
    _replay_case(S, oracle_mod, X, hard, [11, 12, 13, 0], burn, samp)


@pytest.mark.parametrize("shape", EDGE_SHAPES)
def test_replay_bit_exact_edge_shapes(S, oracle_mod, shape):
    rng = np.random.default_rng(hash(shape) & 0xffff)
    X, hard = random_dataset(rng, *shape)
    _replay_case(S, oracle_mod, X, hard, [1, 2, 3], 10, 10)


@pytest.mark.parametrize("name", NOW)
def test_replay_of_unmodified_reference_traces(S, name):
    """Golden fixtures recorded from the UNMODIFIED reference binary (tools/make_golden.py)."""
    g = np.load(os.path.join(GOLDEN, f"ref_{name}.npz"))
    X, hard = load_hex_dataset(name)
    burn, samp = int(g["meta"][0]), int(g["meta"][1])
    run = S.Run(S.Dataset.from_bits(X, hard), 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=burn + samp)
    run.set_tapes([g["tape"]]).init()
    for r in range(len(g["kind"])):
        if r:
            run.advance(1, True)
        st = run.state(0)
        for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
            assert np.array_equal(st[k], g[k][r].astype(np.int32)), (k, r)
        assert st["slots"] == int(g["slots"][r])
        assert st["c"] == g["cdl"][r][0] and st["d"] == g["cdl"][r][1]
        if r:   # after every mcmc_sample(): the saved value, bit-exact; the initial one within 1e-9 relative
            assert st["loglik"] == g["cdl"][r][2], r
        else:
            assert abs(st["loglik"] - g["cdl"][r][2]) <= LL_RTOL * abs(g["cdl"][r][2])
    assert run.state(0)["slots"] == g["tape"].size
    run.close()


def test_replay_100_chains_g10s2(S, oracle_mod):
    """BASELINE.json config 2 at reduced length: 100 chains of g10s2, seeds 0..99."""
    X, hard = load_hex_dataset("g10s2")
    _replay_case(S, oracle_mod, X, hard, list(range(100)), 1, 2)


@pytest.mark.parametrize("name,burn,samp", [("g10s10", 10, 10), ("g2s2", 2, 3)])
def test_free_running_equals_oracle_philox(S, oracle_mod, name, burn, samp):
    X, hard = load_hex_dataset(name)
    seed, offset, n = 20060206, 40, 6
    run = S.Run(S.Dataset.from_bits(X, hard), n, mode=S.MODE_FREE, seed=seed, chain_offset=offset,
                store=S.STORE_FULL, max_samples=samp)
    run.init().advance(burn, False).advance(samp, True).sync()
    assert run.check() == 0
    for i in range(n):
        o, init, res, final, tape = _oracle_chain(oracle_mod, X, hard, 0, burn, samp, philox=(seed, offset + i), detmath=True)
        got = run.state(i)
        for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
            assert np.array_equal(got[k], getattr(final, k)), (i, k)
        assert got["c"] == final.c and got["d"] == final.d
        _cmp_samples(run.fetch_samples(i), res, ("free", i))
    run.close()


def test_sharding_is_invisible(S):
    """Chains keyed by GLOBAL id: 8 chains in one run == two runs of 4 with chain_offset."""
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    whole = S.Run(ds, 8, seed=5, store=S.STORE_PI, max_samples=3).init().advance(3, False).advance(3, True).sync()
    parts = [S.Run(ds, 4, seed=5, chain_offset=o, store=S.STORE_PI, max_samples=3).init().advance(3, False).advance(3, True).sync()
             for o in (0, 4)]
    for i in range(8):
        a, b = whole.state(i), parts[i // 4].state(i % 4)
        for k in ("a", "b", "pi", "tot"):
            assert np.array_equal(a[k], b[k])
        assert a["loglik"] == b["loglik"]


def test_selection_and_pair_order_on_device(S, oracle_mod):
    X, hard = load_hex_dataset("g10s10")
    n, samp, k = 64, 12, 4
    run = S.Run(S.Dataset.from_bits(X, hard), n, seed=7, store=S.STORE_PI, max_samples=samp)
    run.init().advance(20, False).advance(samp, True).sync()
    e = run.chain_stats()["e_negloglik"]
    import torch
    d_e = torch.empty(n, dtype=torch.float64, device="cuda")
    d_ch = torch.empty(k, dtype=torch.int32, device="cuda")
    d_info = torch.empty(3, dtype=torch.float64, device="cuda")
    run.chain_stats_device(d_e.data_ptr())
    run.sync()
    assert np.array_equal(d_e.cpu().numpy(), e)
    S.select_chains_device(d_e.data_ptr(), n, k, d_ch.data_ptr(), d_info.data_ptr())
    torch.cuda.synchronize()
    want = oracle_mod.choose_chains(e, k)
    got = [int(v) for v in d_ch.cpu().numpy() if v >= 0]
    assert got == want and int(d_info[0].item()) == len(want)
    assert d_info[1].item() == e.min() and abs(d_info[2].item() - np.std(e)) < 1e-9
    assert list(S.select_chains(e, k)[0]) == want
    counts = run.po_counts(want)
    for c, ch in enumerate(want):
        pis = run.fetch_samples(ch, full=False)["pi"]
        assert np.array_equal(counts[c], oracle_mod.pair_order_counts(pis))
    po = S.po_finalize(counts, k)
    ref = oracle_mod.pair_order_matrix([oracle_mod.pair_order_counts(run.fetch_samples(ch, full=False)["pi"]) for ch in want], k)
    assert np.max(np.abs(po - ref)) < 1e-12


def test_invariants_at_scale_g2s2(S):
    """mcmc_consistent on every chain of a 2048-chain g2s2 batch (size-independent property)."""
    X, hard = load_hex_dataset("g2s2")
    run = S.Run(S.Dataset.from_bits(X, hard), 2048, seed=1).init().advance(3, False).advance(2, True).sync()
    assert run.check() == 0
    st = run.chain_stats()
    assert st["n_samples"] == 2 and np.all(st["e_negloglik"] > 0) and np.all((st["e_c"] > .001) & (st["e_c"] < .1))


def test_error_paths(S):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    with pytest.raises(S.SeriationError):
        S.Run(ds, 2).advance(1, False)                      # advance before init
    with pytest.raises(S.SeriationError):
        S.Run(ds, 2, mode=S.MODE_REPLAY).init()             # replay without tapes
    short = S.Run(ds, 1, mode=S.MODE_REPLAY).set_tapes([np.full(300, 0.5)]).init().advance(1, False).sync()
    with pytest.raises(S.SeriationError) as e:
        short.state(0)                                      # tape exhausted mid-run
    assert "tape" in str(e.value)
    with pytest.raises(S.SeriationError) as e:
        S.Run(S.Dataset.from_bits(np.ones((4, 9000), np.uint8)), 1)  # unsupported shape says so
    assert "M=9000" in str(e.value)
    with pytest.raises(S.SeriationError):
        S.Run(S.Dataset.from_bits(np.ones((2049, 3), np.uint8)), 1)


def test_reference_file_writers(S, oracle_mod, tmp_path):
    """Chains/chain_XX/ files: same layout and numbers as the reference's writers (mcmc.c:69-92,
    :60-67, :261-294), checked by parsing them the way script.py does."""
    X, hard = load_hex_dataset("g10s10")
    o, init, res, final, tape = _oracle_chain(oracle_mod, X, hard, 21, 3, 5)
    run = S.Run(S.Dataset.from_bits(X, hard), 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=5)
    run.set_tapes([tape]).init().advance(3, False).advance(5, True).sync()
    run.write_chain_files(0, str(tmp_path))
    lines = (tmp_path / "chain_data.csv").read_text().split("\n")
    assert len(lines) == 6 and lines[-1] == ""
    N, M = X.shape
    for s, line in enumerate(lines[:5]):
        f = line.split(",")
        assert [int(v) for v in f[0].split()] == res["a"][s].tolist()
        assert [int(v) for v in f[1].split()] == res["b"][s].tolist()
        assert [int(v.strip()) for v in f[2].split(" ")[:N]] == res["pi"][s].tolist()  # script.py:144-145
        assert f[3].split(" ")[0] == "%.14f" % np.exp(res["c"][s]) and len(f[3].split()) == M
        assert f[4].split(" ")[0] == "%.14f" % np.exp(res["d"][s])
        assert abs(float(f[5]) - res["loglik"][s]) <= LL_RTOL * abs(res["loglik"][s])
    exp = (tmp_path / "exp_data.csv").read_text().split("\n")
    assert exp[0] == "exp_loglik,exp_c,exp_d" and len(exp) == 2
    vals = [float(v) for v in exp[1].split(",")]
    assert abs(vals[0] - res["sums"][0] / 1000) < 1e-9 and abs(vals[1] - res["sums"][1] / 1000) < 1e-13
    taxa = (tmp_path / "taxa.csv").read_text().split("\n")
    assert taxa[0] == "a,b,c,d" and taxa[1].startswith("%d,%d," % (final.a[0], final.b[0]))
    sites = (tmp_path / "sites.csv").read_text().split("\n")
    assert sites[0] == "sites" and [int(v) for v in sites[1:N + 1]] == final.pi.tolist()
    hs = (tmp_path / "hard_sites.csv").read_text().split("\n")
    assert hs[0] == "i,pi_i" and len(hs) == int(hard.sum()) + 2


def test_cli_drop_in_full_length_vs_reference_cli(S, oracle_mod, tmp_path):
    """`mcmc 7 < g10s10.txt`, the call script.py:44-45 makes: the UNMODIFIED reference main() with GSL_RNG_SEED=7
    (1000 + 1000 calls = 20 000 sweeps, files under Chains/chain_07/) left E[-logL] = tests/golden/ref_free_g10s10.npz's
    e_negloglik[7] in its exp_data.csv (tools/make_golden_free.py).  This repo's `mcmc` replays the shim's MT19937 stream of
    that seed (regenerated by the oracle, tests/test_oracle_vs_ref.py) and must print the same number; its chain_data.csv
    carries the oracle's 1000 samples."""
    import subprocess
    from tools.datasets import write_txt
    g = np.load(os.path.join(GOLDEN, "ref_free_g10s10.npz"))
    X, hard = load_hex_dataset("g10s10")
    ds = tmp_path / "g10s10.txt"
    write_txt(str(ds), X, hard)
    o, init, res, final, tape = _oracle_chain(oracle_mod, X, hard, 7, 1000, 1000)
    tape_path = tmp_path / "tape.bin"
    tape.tofile(str(tape_path))
    env = dict(os.environ, SER_TAPE_IN=str(tape_path))
    env.pop("GSL_RNG_SEED", None)
    with open(ds) as f:
        subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "7"], stdin=f, cwd=tmp_path, env=env, check=True)
    out = tmp_path / "Chains" / "chain_07"
    exp = (out / "exp_data.csv").read_text().split("\n")
    assert exp[0] == "exp_loglik,exp_c,exp_d"
    assert float(exp[1].split(",")[0]) == g["e_negloglik"][7]
    lines = (out / "chain_data.csv").read_text().split("\n")
    assert len(lines) == 1001
    for s in (0, 499, 999):
        f = lines[s].split(",")
        assert [int(v) for v in f[0].split()] == res["a"][s].tolist() and [int(v) for v in f[1].split()] == res["b"][s].tolist()
        assert [int(v.strip()) for v in f[2].split(" ")[:X.shape[0]]] == res["pi"][s].tolist()
    assert [int(v) for v in (out / "sites.csv").read_text().split("\n")[1:X.shape[0] + 1]] == final.pi.tolist()


def test_cli_batch_mode(S, tmp_path):
    import subprocess
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    ds = tmp_path / "g10s10.txt"
    write_txt(str(ds), X, hard)
    out = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "12", "--burn", "20", "--samples", "10", "--seed", "9",
                          "--dataset", str(ds), "--chains-dir", str(tmp_path / "Chains"), "--select", "3",
                          "--po", str(tmp_path / "po.csv")], check=True, capture_output=True, text=True).stdout
    assert "selection:" in out and "sweeps/s" in out
    assert sorted(os.listdir(tmp_path / "Chains")) == ["chain_%02d" % i for i in range(12)]
    po = np.loadtxt(tmp_path / "po.csv", delimiter=",")
    assert po.shape == (124, 124) and np.all(np.diag(po) < 0)
    # the same chains through the Python mirror of script.py
    batch = S.run_all_chains(str(ds), 12, 20, 10, seed=9)
    e = batch.stats()["e_negloglik"]
    first = float((tmp_path / "Chains" / "chain_00" / "exp_data.csv").read_text().split("\n")[1].split(",")[0])
    assert abs(first - e[0] * 10 / 1000) < 1e-6   # print_exp_data divides by the literal 1000
    chosen = S.choose_chains(batch, 3)
    assert ("chosen " + " ".join(str(c) for c in chosen)) in out
    assert np.allclose(S.compute_pair_order_matrix(batch, chosen, 3), po, atol=1e-6)


# ------------------------------------------------------------------------------------------------
# large-shape path (ser_sweep_kernel_big): several columns per thread, bit columns / items in
# L2-resident global scratch.  SER_FORCE_BIG=<threads> routes small shapes through it.
@pytest.mark.parametrize("warp", ["0", "1"])
@pytest.mark.parametrize("threads", ["64", "1024"])
@pytest.mark.parametrize("name,burn,samp", [("g10s10", 8, 8), ("g2s2", 2, 2)])
def test_big_path_replay_bit_exact(S, oracle_mod, monkeypatch, name, burn, samp, threads, warp):
    """both forms of the Gibbs phase: CTA-wide column groups (SER_BIG_WARP=0) and warp batches (the default when every
    column's items fit a warp's slice of the item buffers)"""
    monkeypatch.setenv("SER_FORCE_BIG", threads)
    monkeypatch.setenv("SER_BIG_WARP", warp)
    X, hard = load_hex_dataset(name)
    probe = S.Run(S.Dataset.from_bits(X, hard), 1)
    assert probe.kernel_path() == (2 if warp == "1" else 1)
    probe.close()
    _replay_case(S, oracle_mod, X, hard, [5, 6, 7], burn, samp)


def test_big_path_warp_batches_fall_back_when_a_column_is_too_wide(S, oracle_mod, monkeypatch):
    """a full column of 700 sites = 701 items does not fit a warp's slice at 1024 threads / 100 KB: the CTA-wide groups serve
    the shape; with 64 threads the slice is large enough and the warp batches do"""
    rng = np.random.default_rng(5)
    X = (rng.random((700, 40)) < 0.2).astype(np.uint8)
    X[:, 3] = 1
    hard = np.zeros(700, np.uint8); hard[[10, 300, 650]] = 1
    monkeypatch.setenv("SER_BIG_SMEM_KB", "100")
    for threads, path in (("1024", 1), ("64", 2)):
        monkeypatch.setenv("SER_FORCE_BIG", threads)
        probe = S.Run(S.Dataset.from_bits(X, hard), 1)
        assert probe.kernel_path() == path
        probe.close()
        _replay_case(S, oracle_mod, X, hard, [1, 2], 3, 3)


@pytest.mark.parametrize("threads,kb", [("256", "40"), ("1024", "48"), ("320", "64")])
def test_big_path_small_budget_replay_bit_exact(S, oracle_mod, monkeypatch, threads, kb):
    """the large-shape Gibbs phase with a small shared-memory budget: several column groups per step even on the NOW subsets"""
    monkeypatch.setenv("SER_FORCE_BIG", threads)
    monkeypatch.setenv("SER_BIG_SMEM_KB", kb)
    for name, burn, samp in (("g10s10", 6, 6), ("g2s2", 2, 2)):
        X, hard = load_hex_dataset(name)
        _replay_case(S, oracle_mod, X, hard, [5, 6, 7], burn, samp)
    X, hard = load_hex_dataset("g5s5")
    _manycd_replay_case(S, oracle_mod, X, hard, [3], 3, 3)


@pytest.mark.parametrize("shape", EDGE_SHAPES[::2])
def test_big_path_edge_shapes(S, oracle_mod, monkeypatch, shape):
    monkeypatch.setenv("SER_FORCE_BIG", "32")
    rng = np.random.default_rng(hash(shape) & 0xffff)
    X, hard = random_dataset(rng, *shape)
    _replay_case(S, oracle_mod, X, hard, [1, 2], 6, 6)


def test_big_path_many_chains_share_slots(S, oracle_mod, monkeypatch):
    """more chains than resident CTA slots: the persistent grid walks over chains"""
    monkeypatch.setenv("SER_FORCE_BIG", "1024")
    X, hard = load_hex_dataset("g10s10")
    run = S.Run(S.Dataset.from_bits(X, hard), 700, seed=3, store=S.STORE_PI, max_samples=2)
    run.init().advance(2, False).advance(2, True).sync()
    assert run.check() == 0
    monkeypatch.delenv("SER_FORCE_BIG")
    ref = S.Run(S.Dataset.from_bits(X, hard), 700, seed=3, store=S.STORE_PI, max_samples=2)
    ref.init().advance(2, False).advance(2, True).sync()
    for i in (0, 1, 147, 148, 149, 400, 699):
        a, b = run.state(i), ref.state(i)
        for k in ("a", "b", "pi", "tot"):
            assert np.array_equal(a[k], b[k]), (i, k)
        assert a["loglik"] == b["loglik"]


def test_wide_matrix_uses_big_path_replay(S, oracle_mod):
    """M > 1023 (more taxa than threads in a CTA): synthetic 200 x 1500"""
    X, hard = S.Dataset.synthetic(200, 1500, 6, 11).arrays()
    _replay_case(S, oracle_mod, X, hard, [1, 2], 2, 2)


def test_synthetic_1024x4096_replay(S, oracle_mod):
    """BASELINE.json config 5 shape: 1024 sites x 4096 taxa, one chain, 10 + 10 sweeps vs the oracle"""
    X, hard = S.Dataset.synthetic(1024, 4096, 16).arrays()
    _replay_case(S, oracle_mod, X, hard, [42], 1, 1)
    run = S.Run(S.Dataset.from_bits(X, hard), 300, seed=1).init().advance(1, False).advance(1, True).sync()
    assert run.check() == 0 and run.kernel_path() == 2


def test_synthetic_1024x4096_groups_equal_warp_batches(S, monkeypatch):
    """the two forms of the large-shape Gibbs phase on the config-5 shape, free-running: identical chains"""
    ds = S.Dataset.synthetic(1024, 4096, 16)
    fp = []
    for warp in ("1", "0"):
        monkeypatch.setenv("SER_BIG_WARP", warp)
        run = S.Run(ds, 160, seed=77, store=S.STORE_PI, max_samples=2).init().advance(1, False).advance(2, True).sync()
        assert run.check() == 0 and run.kernel_path() == (2 if warp == "1" else 1)
        fp.append([(run.state(i)["a"].tobytes(), run.state(i)["b"].tobytes(), run.state(i)["pi"].tobytes(), run.state(i)["loglik"])
                   for i in (0, 1, 147, 148, 159)])
        run.close()
    assert fp[0] == fp[1]


def test_config3_g5s5_4096_chains_selection_and_po(S, oracle_mod):
    """BASELINE.json config 3 at reduced length: g5s5, 4096 chains, k = 2 (script.py:455-456).
    Device selection == script.py's choose_chains on the same E[-logL]; PO counts == numpy on the
    chosen chains' pi history; and two of the 4096 chains are re-run on the CPU oracle (same Philox
    stream) to tie the batch back to the reference algorithm."""
    X, hard = load_hex_dataset("g5s5")
    n, burn, samp, k, seed = 4096, 6, 8, 2, 20060206
    run = S.Run(S.Dataset.from_bits(X, hard), n, seed=seed, store=S.STORE_PI, max_samples=samp)
    run.init().advance(burn, False).advance(samp, True).sync()
    assert run.check() == 0
    st = run.chain_stats()
    e = st["e_negloglik"]
    want = oracle_mod.choose_chains(e, k)
    assert list(S.select_chains(e, k)[0]) == want and len(want) == k
    counts = run.po_counts(want)
    for c, ch in enumerate(want):
        assert np.array_equal(counts[c], oracle_mod.pair_order_counts(run.fetch_samples(ch, full=False)["pi"]))
    po = S.po_finalize(counts, k)
    assert po.shape == (273, 273) and np.all(np.diag(po) < 0)
    for ch in (want[0], 4095):
        o, init, res, final, tape = _oracle_chain(oracle_mod, X, hard, 0, burn, samp, philox=(seed, ch), detmath=True)
        assert np.array_equal(run.fetch_samples(ch, full=False)["pi"], res["pi"])
        assert abs(e[ch] - res["sums"][0] / samp) <= LL_RTOL * e[ch]


def test_free_running_reproduces_report_table1_g10s10(S):
    """End-to-end statistical check against the reference's published result (Docs/Report.pdf
    Table 1, g10s10: E[c] = 0.0119, E[d] = 0.5127 over the 8 best of 100 chains; 10k burn-in +
    10k sampling sweeps, thin 10).  Free-running Philox chains, full length."""
    X, hard = load_hex_dataset("g10s10")
    run = S.Run(S.Dataset.from_bits(X, hard), 100, seed=12345, store=S.STORE_PI, max_samples=1000)
    run.init().advance(1000, False).advance(1000, True).sync()
    assert run.check() == 0
    st = run.chain_stats()
    chosen, mn, sd = S.select_chains(st["e_negloglik"], 8)
    assert len(chosen) == 8
    e_c, e_d = st["e_c"][chosen].mean(), st["e_d"][chosen].mean()
    assert abs(e_c - 0.0119) < 0.003, e_c
    assert abs(e_d - 0.5127) < 0.05, e_d
    # the seriation itself: expected correlation of the order with the file order (MN age order), 0.94 in the report
    pis = np.concatenate([run.fetch_samples(int(c), full=False)["pi"] for c in chosen])
    corr = np.mean([abs(np.corrcoef(p, np.arange(p.size))[0, 1]) for p in pis[::50]])
    assert corr > 0.85, corr


def test_launch_splitting_is_invisible(S):
    """advance(n) == n x advance(1): the chain state carried through HBM between launches is complete"""
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    one = S.Run(ds, 5, seed=77, store=S.STORE_FULL, max_samples=6).init().advance(4, False).advance(6, True).sync()
    many = S.Run(ds, 5, seed=77, store=S.STORE_FULL, max_samples=6).init()
    for c in range(10):
        many.advance(1, c >= 4)
    many.sync()
    for i in range(5):
        a, b = one.state(i), many.state(i)
        for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
            assert np.array_equal(a[k], b[k]), (i, k)
        assert (a["c"], a["d"], a["loglik"]) == (b["c"], b["d"], b["loglik"])
        sa, sb = one.fetch_samples(i), many.fetch_samples(i)
        assert all(np.array_equal(sa[k], sb[k]) for k in sa)
    assert np.array_equal(one.chain_stats()["e_negloglik"], many.chain_stats()["e_negloglik"])
    assert np.array_equal(one.counters(0), many.counters(0)) and one.counters(0)[7] == 100


def test_sample_store_capacity_and_modes(S):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    run = S.Run(ds, 2, seed=1, store=S.STORE_PI, max_samples=3).init().advance(5, True).sync()
    assert run.chain_stats()["n_samples"] == 5              # the exp_data sums keep running ...
    assert run.fetch_samples(0, full=False)["pi"].shape == (3, 124)   # ... the store keeps the first max_samples
    with pytest.raises(S.SeriationError):
        run.fetch_samples(0, full=True)                      # a, b, c, d were not stored
    none = S.Run(ds, 2, seed=1).init().advance(2, True).sync()
    with pytest.raises(S.SeriationError):
        none.po_counts([0])                                  # no pi history without SER_STORE_PI
    assert none.chain_stats()["n_samples"] == 2


def test_posterior_summaries_on_device(S, oracle_mod):
    """SURVEY section 8f #1: compute_exp_ages / compute_exp_pi / compute_exp_a over the GPU's sample store"""
    X, hard = load_hex_dataset("g10s10")
    batch = S.run_all_chains(S.Dataset.from_bits(X, hard), 24, 30, 16, seed=4, store=S.STORE_FULL)
    chains = S.choose_chains(batch, 3)
    assert len(chains) == 3
    samples = [batch.run.fetch_samples(c) for c in chains]
    ps = batch.run.posterior_sums(chains, with_ab=True)
    assert ps["n_samples"] == 16
    for slot, smp in enumerate(samples):
        assert np.array_equal(ps["pi_sum"][slot], smp["pi"].sum(axis=0))
        assert np.array_equal(ps["a_sum"][slot], smp["a"].sum(axis=0)) and np.array_equal(ps["b_sum"][slot], smp["b"].sum(axis=0))
        assert ps["corr_num"][slot] == int((smp["pi"] * np.arange(124)).sum())
    pis, a_s = [s["pi"] for s in samples], [s["a"] for s in samples]
    assert abs(S.compute_exp_ages(batch, chains, 3, 124) - oracle_mod.exp_ages(pis, 3)) < 1e-12
    assert np.allclose(S.compute_exp_pi(batch, chains, 124, 3), oracle_mod.exp_pi(pis, 3), rtol=0, atol=1e-12)
    assert np.allclose(S.compute_exp_a(batch, chains, 3, 139), oracle_mod.exp_a(a_s, 3), rtol=0, atol=1e-12)
    exp_c, exp_d = S.compute_exp_cd(batch, chains, 3, faithful=False)
    assert 0.001 < exp_c < 0.1 and 0.2 < exp_d < 0.8


def test_labelled_outputs(S, tmp_path):
    X = (np.random.default_rng(2).random((12, 5)) < .4).astype(np.uint8)
    hard = np.zeros(12, np.uint8); hard[[2, 9]] = 1
    ds = S.Dataset.from_bits(X, hard)
    (tmp_path / "t.genus").write_text("".join("Genus_%d \n" % m for m in range(5)))
    (tmp_path / "t.sites").write_text("".join("Site_%d [%d,%.2f]%s\n" % (n, n // 3, 20 - n, " *" if hard[n] else "") for n in range(12)))
    run = S.Run(ds, 1, seed=3).init().advance(3, False).sync()
    with pytest.raises(S.SeriationError):
        run.write_labelled_files(0, str(tmp_path))            # no labels yet
    ds.read_names(str(tmp_path / "t.genus"), str(tmp_path / "t.sites"))
    run.write_labelled_files(0, str(tmp_path))
    st = run.state(0)
    taxa = (tmp_path / "taxa_named.csv").read_text().split("\n")
    assert taxa[0] == "taxon,a,b" and taxa[1] == "Genus_0,%d,%d" % (st["a"][0], st["b"][0])
    sites = (tmp_path / "sites_named.csv").read_text().split("\n")
    assert sites[3] == "Site_2,0,18,1,%d" % st["pi"][2]


# ----------------------------------------------------------------------------- per-taxon c, d (manycd = 1)
def _manycd_oracle(O, X, hard, seed=None, philox=None, tape=None, detmath=False):
    o = O.Oracle(X, hard).manycd()
    if tape is not None:
        o.source_tape(tape)
    elif philox is not None:
        o.source_philox(*philox)
    else:
        o.source_mt(seed)
    o.record(True).detmath(detmath)
    o.randomize()
    return o


def _cmp_manycd(run, i, want, what, exact_ll):
    got = run.state(i)
    for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
        assert np.array_equal(got[k], getattr(want, k)), (what, k)
    c, d = run.cd(i)
    assert c.tobytes() == want.c_all.tobytes() and d.tobytes() == want.d_all.tobytes(), what
    assert got["c"] == want.c_all[0] and got["d"] == want.d_all[0], what
    if exact_ll:
        assert got["loglik"] == want.loglik, (what, got["loglik"], want.loglik)
    else:
        assert abs(got["loglik"] - want.loglik) <= LL_RTOL * abs(want.loglik), what


def _manycd_replay_case(S, O, X, hard, seeds, burn, samp):
    oracles = [_manycd_oracle(O, X, hard, seed=s) for s in seeds]
    inits = [o.state() for o in oracles]
    trace = []
    for o in oracles:   # record the tapes first: the run needs them whole
        trace.append([o.sample() and None or o.state() for _ in range(burn + samp)])
    run = S.Run(S.Dataset.from_bits(X, hard), len(seeds), mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=samp, manycd=True)
    run.set_tapes([o.tape() for o in oracles]).init().sync()
    for i in range(len(seeds)):
        _cmp_manycd(run, i, inits[i], ("init", i), False)
    run.advance(burn, False).sync()
    for i in range(len(seeds)):
        _cmp_manycd(run, i, trace[i][burn - 1], ("burn", i), False)
    for s in range(samp):
        run.advance(1, True).sync()
        for i in range(len(seeds)):
            _cmp_manycd(run, i, trace[i][burn + s], ("sample", s, i), True)
    assert run.check() == 0
    for i, o in enumerate(oracles):
        assert run.state(i)["slots"] == o.tape().size
        got = run.fetch_samples(i)
        for s in range(samp):
            w = trace[i][burn + s]
            assert np.array_equal(got["a"][s], w.a) and np.array_equal(got["b"][s], w.b) and np.array_equal(got["pi"][s], w.pi)
            assert got["c_all"][s].tobytes() == w.c_all.tobytes() and got["d_all"][s].tobytes() == w.d_all.tobytes()
            assert got["c"][s] == w.c_all[0] and got["d"][s] == w.d_all[0] and got["loglik"][s] == w.loglik
    run.close()


@pytest.mark.parametrize("name,burn,samp", [("g10s10", 20, 20), ("g5s5", 3, 3), ("g2s2", 3, 3)])
def test_manycd_replay_bit_exact(S, oracle_mod, name, burn, samp):
    X, hard = load_hex_dataset(name)
    _manycd_replay_case(S, oracle_mod, X, hard, [31, 32, 0], burn, samp)


@pytest.mark.parametrize("shape", EDGE_SHAPES)
def test_manycd_replay_edge_shapes(S, oracle_mod, shape):
    rng = np.random.default_rng(hash(shape) & 0xffff)
    X, hard = random_dataset(rng, *shape)
    _manycd_replay_case(S, oracle_mod, X, hard, [4, 5], 8, 8)


def test_manycd_replay_of_unmodified_reference_trace(S):
    """golden trace of the UNMODIFIED reference run as `mcmc 1 tb ts` (tools/make_golden.py)"""
    g = np.load(os.path.join(GOLDEN, "ref_g10s10_manycd.npz"))
    X, hard = load_hex_dataset("g10s10")
    run = S.Run(S.Dataset.from_bits(X, hard), 1, mode=S.MODE_REPLAY, manycd=True)
    run.set_tapes([g["tape"]]).init()
    for r in range(len(g["kind"])):
        if r:
            run.advance(1, True)
        st = run.state(0)
        for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
            assert np.array_equal(st[k], g[k][r].astype(np.int32)), (k, r)
        assert st["slots"] == int(g["slots"][r])
        c, d = run.cd(0)
        assert c.tobytes() == g["c_all"][r].tobytes() and d.tobytes() == g["d_all"][r].tobytes(), r
        if r:
            assert st["loglik"] == g["cdl"][r][2], r
        else:
            assert abs(st["loglik"] - g["cdl"][r][2]) <= LL_RTOL * abs(g["cdl"][r][2])
    run.close()


@pytest.mark.parametrize("name,burn,samp", [("g10s10", 10, 10), ("g2s2", 2, 2)])
def test_manycd_free_running_equals_oracle_philox(S, oracle_mod, name, burn, samp):
    X, hard = load_hex_dataset(name)
    seed, offset, n = 1234, 17, 4
    run = S.Run(S.Dataset.from_bits(X, hard), n, mode=S.MODE_FREE, seed=seed, chain_offset=offset, manycd=True)
    run.init().advance(burn, False).advance(samp, True).sync()
    assert run.check() == 0
    for i in range(n):
        o = _manycd_oracle(oracle_mod, X, hard, philox=(seed, offset + i), detmath=True)
        for _ in range(burn + samp):
            o.sample()
        _cmp_manycd(run, i, o.state(), ("free", i), True)
    run.close()


def test_manycd_errors_and_writers(S, oracle_mod, tmp_path):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    wide = S.Run(S.Dataset.from_bits(np.ones((8, 2000), np.uint8)), 1, manycd=True).init().advance(1, True).sync()
    assert wide.check() == 0 and len(set(wide.cd(0)[0])) > 100   # more taxa than threads: the large-shape per-taxon instantiation
    wide.close()
    plain = S.Run(ds, 1).init()
    with pytest.raises(S.SeriationError):
        plain.cd(0)
    plain.close()
    o = _manycd_oracle(oracle_mod, X, hard, seed=3)
    states = [o.sample() and None or o.state() for _ in range(6)]
    run = S.Run(ds, 1, mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=4, manycd=True)
    run.set_tapes([o.tape()]).init().advance(2, False).advance(4, True).sync()
    run.write_chain_files(0, str(tmp_path))
    N, M = X.shape
    lines = (tmp_path / "chain_data.csv").read_text().split("\n")
    for s, line in enumerate(lines[:4]):
        f, w = line.split(","), states[2 + s]
        assert [int(v) for v in f[0].split()] == w.a.tolist()
        assert f[3].split() == ["%.14f" % np.exp(v) for v in w.c_all]   # mcmc.c:86-87 prints exp(c[i]) per taxon
        assert f[4].split() == ["%.14f" % np.exp(v) for v in w.d_all]
        assert f[5] == "%.14f" % w.loglik
    taxa = (tmp_path / "taxa.csv").read_text().split("\n")
    w = states[-1]
    assert taxa[1:M + 1] == ["%d,%d,%.14f,%.14f" % (w.a[i], w.b[i], np.exp(w.c_all[i]), np.exp(w.d_all[i])) for i in range(M)]
    run.close()


def test_manycd_cli(S, oracle_mod, tmp_path):
    """`mcmc 1 3 4 < g10s10.txt` (manycd Tburnin T, mcmc.c:115-121).  The unmodified reference cannot
    finish this form -- chain_index stays NULL and atoi(NULL) faults at mcmc.c:153 -- so the files are
    checked against the oracle (itself pinned to the reference's manycd sampler by the golden trace)."""
    import subprocess
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    N, M = X.shape
    ds = tmp_path / "g10s10.txt"
    write_txt(str(ds), X, hard)
    o = _manycd_oracle(oracle_mod, X, hard, seed=77)
    states = [o.sample() and None or o.state() for _ in range(7)]
    tape = tmp_path / "tape.bin"
    o.tape().tofile(str(tape))
    env = dict(os.environ, SER_TAPE_IN=str(tape))
    with open(ds) as f:
        subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "1", "3", "4"], stdin=f, cwd=tmp_path, env=env, check=True)
    out = tmp_path / "Chains" / "chain_00"
    lines = (out / "chain_data.csv").read_text().split("\n")
    assert len(lines) == 5
    for s, line in enumerate(lines[:4]):
        f, w = line.split(","), states[3 + s]
        assert [int(v) for v in f[1].split()] == w.b.tolist() and [int(v) for v in f[2].split()] == w.pi.tolist()
        assert f[3].split() == ["%.14f" % np.exp(v) for v in w.c_all] and f[5] == "%.14f" % w.loglik
    w = states[-1]
    assert (out / "taxa.csv").read_text().split("\n")[M] == "%d,%d,%.14f,%.14f" % (w.a[M - 1], w.b[M - 1], np.exp(w.c_all[M - 1]), np.exp(w.d_all[M - 1]))


# ----------------------------------------------------------------------------- script.py's analysis, end to end
def test_script_mirror_equals_unmodified_script_py(S):
    """tests/golden/script_g10s10.npz holds what the UNMODIFIED script.py computed (choose_chains,
    compute_exp_cd, compute_exp_ages, compute_pair_order_matrix, compute_exp_pi, compute_exp_a and the three
    probability maps) over a Chains/ directory of 6 Philox chains; the GPU free-running mode
    reproduces those chains, and the Python mirror over the device reductions must give the same numbers."""
    g = np.load(os.path.join(GOLDEN, "script_g10s10.npz"))
    seed, n_chains, burn, samp, k = (int(v) for v in g["meta"])
    X, hard = load_hex_dataset("g10s10")
    N, M = X.shape
    batch = S.run_all_chains(S.Dataset.from_bits(X, hard), n_chains, burn, samp, seed=seed, store=S.STORE_FULL)
    # exp_data.csv divides by the literal 1000 (mcmc.c:65); the mirror's E[-logL] divides by the samples taken
    e = batch.stats()["e_negloglik"]
    for i in range(n_chains):
        assert e[i] == float(g["e_negloglik_%d" % i]), i
    chosen = S.choose_chains(batch, k)
    assert chosen == g["chosen"].tolist()
    ec, ed = S.compute_exp_cd(batch, chosen, k)
    # the reference sums the %.14f-printed values and divides by the literal 1000 (script.py:119-120); so does the mirror
    assert abs(ec - g["exp_cd"][0]) < 1e-13 and abs(ed - g["exp_cd"][1]) < 1e-13
    assert abs(S.compute_exp_ages(batch, chosen, k, N) - float(g["exp_ages"])) < 1e-12
    assert np.allclose(S.compute_pair_order_matrix(batch, chosen, k, N), g["po"], rtol=0, atol=1e-15)
    assert np.allclose(S.compute_exp_pi(batch, chosen, N, k), g["exp_pi"], rtol=0, atol=1e-13)
    assert np.allclose(S.compute_exp_a(batch, chosen, k, M), g["exp_a"], rtol=0, atol=1e-13)
    assert np.allclose(S.taxa_occurence_probability_matrix(batch, chosen, k, N, M), g["alive"], rtol=0, atol=1e-15)
    assert np.allclose(S.false_taxa_occurence_probability_matrix(batch, chosen, k, N, M), g["false_taxa"], rtol=0, atol=1e-15)
    assert np.allclose(S.false_ones_probability_matrix(batch, chosen, k, None, N, M), g["false_ones"], rtol=0, atol=1e-15)
    Y = S.new_data_matrix(batch, chosen, k)
    assert Y.shape == (N, M) and Y.sum() == X.sum()
    alive, T = batch.run.alive_counts(np.array([chosen[0], -1], np.int32))
    fs = batch.run.fetch_samples(chosen[0])
    j = np.arange(N)[None, :, None]
    want = ((j >= fs["a"][:, None, :]) & (j <= fs["b"][:, None, :])).sum(axis=0)
    assert T == samp and np.array_equal(alive[0], want) and not alive[1].any()
    batch.run.close()


def test_65536_chains_one_launch_and_batch_size_independence(S):
    """BASELINE.json's largest batch: 65 536 chains in one launch (g10s10 to keep it short).  Every chain
    passes mcmc_consistent, and the last chain of the batch is bit-identical to the same global chain id
    simulated alone -- a chain never depends on the batch it runs in."""
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    big = S.Run(ds, 65536, seed=99, store=S.STORE_PI, max_samples=2).init().advance(1, False).advance(2, True).sync()
    assert big.check() == 0
    e = big.chain_stats()["e_negloglik"]
    assert e.shape == (65536,) and np.all(e > 0) and np.unique(e).size > 60000
    for gid in (0, 31337, 65535):
        one = S.Run(ds, 1, seed=99, chain_offset=gid, store=S.STORE_PI, max_samples=2).init().advance(1, False).advance(2, True).sync()
        a, b = big.state(gid), one.state(0)
        for k in ("a", "b", "pi", "tot"):
            assert np.array_equal(a[k], b[k]), (gid, k)
        assert a["loglik"] == b["loglik"] and a["c"] == b["c"] and a["d"] == b["d"]
        assert np.array_equal(big.fetch_samples(gid, full=False)["pi"], one.fetch_samples(0, full=False)["pi"])
        one.close()
    chosen = S.select_chains(e, 8)[0]
    po = S.po_finalize(big.po_counts(chosen), 8, faithful=False)
    assert po.shape == (124, 124) and np.allclose(po + po.T - np.diag(2 * np.diag(po)), (1 - np.eye(124)) * (2 / 1000), atol=1e-12)
    big.close()


def test_free_running_statistics_vs_unmodified_reference_pipeline(S):
    """north_star check (3).  tests/golden/ref_free_g10s10.npz = the UNMODIFIED reference run end to end
    (tools/make_golden_free.py: 100 x `mcmc <i> < g10s10.txt` with MT19937, then the unmodified script.py's
    choose_chains(8) / compute_pair_order_matrix / compute_exp_cd / compute_exp_ages; it reproduces the
    report's Table 1: E[c] 0.01196, E[d] 0.5121, corr 0.940).  The GPU's free-running chains use another
    random stream, so this is statistical:
      * E[-logL]: every selected chain lies within one reference sigma of the reference's best chain, and
        the selected chains' mean within one sigma of the reference's selected mean (measured: 0.02 sigma);
      * PO matrix: the 8-of-100 estimator itself varies between two runs of the SAME sampler by ~0.35 max /
        ~0.008 mean absolute (measured below between two GPU seeds), so the 0.02 bound is applied to the
        mean absolute difference, and the difference to the reference must not exceed the sampler's own
        seed-to-seed spread by more than half."""
    g = np.load(os.path.join(GOLDEN, "ref_free_g10s10.npz"))
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    ref_e, ref_sel = g["e_negloglik"], g["e_negloglik"][g["chosen"]]
    sigma = ref_e.std()
    pos = []
    for seed in (12345, 777):
        batch = S.run_all_chains(ds, 100, 1000, 1000, seed=seed, store=S.STORE_PI)
        assert batch.run.check() == 0
        e = batch.stats()["e_negloglik"]
        chosen = S.choose_chains(batch, 8)
        assert len(chosen) == 8
        assert np.all(np.abs(e[chosen] - ref_e.min()) < sigma), (e[chosen], ref_e.min(), sigma)
        assert abs(e[chosen].mean() - ref_sel.mean()) < sigma
        assert abs(e.std() - sigma) < 0.25 * sigma            # the spread over the 100 chains is the same population
        ec, ed = S.compute_exp_cd(batch, chosen, 8)
        assert abs(ec - g["exp_cd"][0]) < 0.002 and abs(ed - g["exp_cd"][1]) < 0.03, (ec, ed)
        assert abs(S.compute_exp_ages(batch, chosen, 8, 124) - float(g["exp_ages"])) < 0.01
        pos.append(S.compute_pair_order_matrix(batch, chosen, 8, 124))
        batch.run.close()
    own = np.abs(pos[0] - pos[1]).mean()
    for po in pos:
        d = np.abs(po - g["po"])
        assert d.mean() < 0.02, d.mean()
        assert d.mean() < 1.5 * own, (d.mean(), own)


@pytest.mark.parametrize("groups", ["1", "2", "5", "8"])
def test_column_groups_are_invisible(S, oracle_mod, monkeypatch, groups):
    """SER_SWEEP_GROUPS only changes how many columns' item weights share the buffer at a time: the
    replay stays bit-exact for every group count (scalar and per-taxon c, d)."""
    monkeypatch.setenv("SER_SWEEP_GROUPS", groups)
    X, hard = load_hex_dataset("g5s5")
    _replay_case(S, oracle_mod, X, hard, [5, 6], 3, 3)
    _manycd_replay_case(S, oracle_mod, X, hard, [7], 2, 2)


def test_live_runs_of_different_shapes_interleave(S):
    """The dynamic shared-memory opt-in belongs to the kernel function, not to a run: a second run on a
    smaller dataset must not break the launches of a live run on a larger one (and vice versa)."""
    runs = []
    for name in ("g2s2", "g10s10", "g5s5"):
        X, hard = load_hex_dataset(name)
        runs.append(S.Run(S.Dataset.from_bits(X, hard), 8, seed=5).init())
    Xm, hm = load_hex_dataset("g10s10")
    runs.append(S.Run(S.Dataset.from_bits(Xm, hm), 4, seed=5, manycd=True).init())
    for _ in range(2):
        for r in runs:
            r.advance(1, True)
    for r in runs:
        r.sync()
        assert r.check() == 0
        r.close()


# ----------------------------------------------------------------------------- round 2: longer replays, config 5 vs the reference
def _oracle_chains_parallel(O, X, hard, seeds, burn, samp):
    """the oracle's chains on all host cores (ctypes releases the GIL inside orc_run)"""
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        return list(ex.map(lambda s: _oracle_chain(O, X, hard, s, burn, samp), seeds))


def _replay_case_parallel(S, O, X, hard, seeds, burn, samp):
    chains = _oracle_chains_parallel(O, X, hard, seeds, burn, samp)
    run = S.Run(S.Dataset.from_bits(X, hard), len(seeds), mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=samp)
    run.set_tapes([c[4] for c in chains]).init().advance_both(burn, samp).sync()
    assert run.check() == 0
    stats = run.chain_stats()
    for i, (o, init, res, final, tape) in enumerate(chains):
        _cmp_state(run.state(i), final, ("final", i))
        assert run.state(i)["slots"] == tape.size and run.state(i)["loglik"] == final.loglik
        _cmp_samples(run.fetch_samples(i), res, ("samples", i))
        assert stats["e_negloglik"][i] == res["sums"][0] / samp
        # every float decision of this tape stayed away from its boundary (see test_oracle_golden.py).  With ~1e7 picks x
        # ~500 CDF steps per chain set the closest approach is expected around 1e-11; the GPU's CDF is good to ~1e-14
        m = o.margins()
        assert m["min_pick"] > 1e-12 and m["min_accept"] > 1e-10, (i, m)
    run.close()


@pytest.mark.parametrize("name", NOW)
def test_replay_2000_sweeps_16_chains_now_subsets(S, oracle_mod, name):
    """16 chains x (1000 burn-in + 1000 sampling) sweeps on every NOW subset: all 100 thinned samples per chain
    (a, b, pi, c, d and the bits of the saved log-likelihood), final state, cursor, exp_data sums."""
    X, hard = load_hex_dataset(name)
    _replay_case_parallel(S, oracle_mod, X, hard, list(range(200, 216)), 100, 100)


def test_replay_config2_100_chains_1000_sweeps(S, oracle_mod):
    """BASELINE.json config 2 (g10s2, 100 chains, seeds 0..99) at 1000 sweeps per chain"""
    X, hard = load_hex_dataset("g10s2")
    _replay_case_parallel(S, oracle_mod, X, hard, list(range(100)), 50, 50)


def test_config5_replay_vs_unmodified_reference_golden(S, oracle_mod):
    """BASELINE.json config 5's matrix against the UNMODIFIED reference: tests/golden/ref_synthetic_1024x4096.npz holds
    the states oracle/_ref/ref_mcmc_big (mcmc.c with MAXS raised, nothing else) went through for 8 seeds x 10
    mcmc_sample() calls = 100 sweeps.  The tapes (53 MB) are regenerated from the seeds by the oracle's MT19937 --
    length and CRC must equal the reference's recorded tapes -- and replayed through the large-shape kernel:
    a, b, pi (the first seed's in full, every seed's by CRC32), c, d and the saved log-likelihood bits of every call,
    totals and cursor at the end."""
    import zlib
    g = np.load(os.path.join(GOLDEN, "ref_synthetic_1024x4096.npz"))
    X, hard = S.Dataset.synthetic(1024, 4096, 16).arrays()
    assert [zlib.crc32(X.tobytes()), zlib.crc32(hard.tobytes())] == g["x_crc"].tolist()
    seeds, calls = [int(s) for s in g["seeds"]], g["a_crc"].shape[1] - 1
    chains = _oracle_chains_parallel(oracle_mod, X, hard, seeds, 0, calls)
    for i, c in enumerate(chains):
        assert c[4].size == int(g["tape_len"][i]) and zlib.crc32(c[4].tobytes()) == int(g["tape_crc"][i]), i

    def same_states(i, k, got, recs):
        """got[j]: chain i's `k` after record recs[j] of the reference"""
        assert [zlib.crc32(v.astype(np.int16).tobytes()) for v in got] == g[k + "_crc"][i][recs].tolist(), (i, k)
        if i < len(g[k]):
            assert np.array_equal(got, g[k][i][recs].astype(np.int32)), (i, k)

    run = S.Run(S.Dataset.from_bits(X, hard), len(seeds), mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls)
    run.set_tapes([c[4] for c in chains]).init().sync()
    for i in range(len(seeds)):
        st = run.state(i)
        for k in ("a", "b", "pi"):
            same_states(i, k, st[k][None], [0])
    run.advance(calls, True).sync()
    assert run.check() == 0
    for i in range(len(seeds)):
        got, st = run.fetch_samples(i), run.state(i)
        for k in ("a", "b", "pi"):
            same_states(i, k, got[k], list(range(1, calls + 1)))
        assert np.array_equal(got["c"], g["cdl"][i][1:, 0]) and np.array_equal(got["d"], g["cdl"][i][1:, 1]), i
        assert np.array_equal(got["loglik"], g["cdl"][i][1:, 2]), (i, np.max(np.abs(got["loglik"] - g["cdl"][i][1:, 2])))
        assert np.array_equal(st["tot"], g["tot"][i][-1]) and st["slots"] == int(g["slots"][i][-1]), i
    run.close()


def test_fuzz_replay_40_cases_all_variants(S):
    """tools/fuzz_replay.py as a driver-visible test: 40 random shapes / densities / hard-site counts, each through the
    one-thread-per-column kernel, the per-taxon c/d instantiation, the large-shape kernel (random block size and
    group budget), a random column-group count, and three free-running variants -- 7 variants per case, bit-exact
    against the oracle.  The differential evidence that the hand-placed barriers of the sweep kernels hold."""
    from tools.fuzz_replay import run_fuzz
    out = run_fuzz(40, seed=2026)
    assert out["passed"], out["failures"][:3]
    assert len(out["refused"]) < 40   # most variants actually ran


def _batch_fingerprint(S, ds, n, seed, burn, samp, **kw):
    run = S.Run(ds, n, seed=seed, store=S.STORE_PI, max_samples=samp, **kw).init().advance_both(burn, samp).sync()
    assert run.check() == 0
    st = run.chain_stats()
    states = [run.state(i) for i in (0, 1, n // 2, n - 1)]
    po = run.po_counts(np.array([0, n // 3, n - 1], np.int32))
    cnt = np.stack([run.counters(i) for i in (0, n - 1)])
    run.close()
    return st, states, po, cnt


def _same_fingerprint(x, y):
    for k in ("e_negloglik", "e_c", "e_d"):
        assert x[0][k].tobytes() == y[0][k].tobytes(), k
    for sa, sb in zip(x[1], y[1]):
        for k in ("a", "b", "pi", "rpi", "t0", "f0", "t1", "f1", "tot"):
            assert np.array_equal(sa[k], sb[k]), k
        assert (sa["c"], sa["d"], sa["loglik"]) == (sb["c"], sb["d"], sb["loglik"])
    assert np.array_equal(x[2], y[2]) and np.array_equal(x[3], y[3])


def test_determinism_across_runs_and_schedules(S, monkeypatch):
    """race evidence without a race detector: the same 4096-chain free-running batch gives identical bits when run
    twice, with other column-group counts, with one-call work items, with an odd number of persistent CTAs (other
    chain -> SM interleavings) and through the large-shape kernel."""
    X, hard = load_hex_dataset("g5s5")
    ds = S.Dataset.from_bits(X, hard)
    base = _batch_fingerprint(S, ds, 4096, 99, 3, 3)
    _same_fingerprint(base, _batch_fingerprint(S, ds, 4096, 99, 3, 3))
    for env in ({"SER_SWEEP_GROUPS": "1"}, {"SER_SWEEP_GROUPS": "4"}, {"SER_CHUNK_CALLS": "1"}, {"SER_SWEEP_SLOTS": "37"},
                {"SER_CHUNK_CALLS": "2", "SER_SWEEP_SLOTS": "1000"}, {"SER_FORCE_BIG": "256"},
                {"SER_FORCE_BIG": "256", "SER_BIG_WARP": "0"}, {"SER_FORCE_BIG": "96", "SER_BIG_SMEM_KB": "64"}):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        _same_fingerprint(base, _batch_fingerprint(S, ds, 4096, 99, 3, 3))
        for k in env:
            monkeypatch.delenv(k)


def test_work_items_of_one_call_with_few_chains(S, oracle_mod, monkeypatch):
    """fewer chains than persistent CTAs and one-call work items: a chain's items run on different SMs back to back,
    each waiting for the previous one's published state (bit columns included) -- still bit-exact vs the oracle"""
    monkeypatch.setenv("SER_CHUNK_CALLS", "1")
    X, hard = load_hex_dataset("g10s10")
    _replay_case(S, oracle_mod, X, hard, [3, 4, 5], 12, 12)
    _manycd_replay_case(S, oracle_mod, X, hard, [6], 4, 4)


def test_advance_both_equals_two_launches(S):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    one = S.Run(ds, 300, seed=8, store=S.STORE_PI, max_samples=4).init().advance_both(5, 4).sync()
    two = S.Run(ds, 300, seed=8, store=S.STORE_PI, max_samples=4).init().advance(5, False).advance(4, True).sync()
    assert one.chain_stats()["e_negloglik"].tobytes() == two.chain_stats()["e_negloglik"].tobytes()
    for i in (0, 150, 299):
        assert np.array_equal(one.fetch_samples(i, full=False)["pi"], two.fetch_samples(i, full=False)["pi"])
        assert one.state(i)["loglik"] == two.state(i)["loglik"]
    assert one.kernel_launches() < two.kernel_launches()


# ----------------------------------------------------------------------------- round 2: the boundary
def test_integration_snippet_runs(S, tmp_path, monkeypatch):
    """INTEGRATION.md's Level-2 ctypes snippet, executed as printed (only the run length is shortened)"""
    from tools.datasets import write_txt
    text = open(os.path.join(os.path.dirname(GOLDEN), "..", "INTEGRATION.md")).read()
    level2 = text[text.index("## Level 2"):]
    snippet = level2[level2.index("```python\n") + len("```python\n"):level2.index("\n```\n")]
    line = "n_chains, burn, samples, k = 4096, 1000, 1000, 2"
    assert line in snippet
    snippet = snippet.replace(line, "n_chains, burn, samples, k = 256, 20, 20, 2")
    (tmp_path / "Dataset").mkdir()
    write_txt(str(tmp_path / "Dataset" / "g10s10.txt"), *load_hex_dataset("g10s10"))
    monkeypatch.chdir(tmp_path)
    monkeypatch.setenv("SERIATION_B200_LIB", S.LIB_PATH)
    ns = {}
    exec(snippet, ns)
    po = np.array(ns["po"][:]).reshape(124, 124)
    assert ns["nk"].value == 2 and np.all(np.diag(po) < 0) and 0 <= ns["chosen"][0] < ns["chosen"][1] < 256
    # the same numbers through the shipped wrapper
    run = S.Run(S.Dataset.from_bits(*load_hex_dataset("g10s10")), 256, seed=20060206, store=S.STORE_PI, max_samples=20)
    res = run.init().advance_both(20, 20).cross_chain(2)
    assert list(res["chosen"]) == list(ns["chosen"][:]) and np.array_equal(S.po_finalize(res["counts"], 2), po)


def test_cross_chain_one_call_equals_the_separate_steps(S, oracle_mod):
    X, hard = load_hex_dataset("g10s10")
    n, samp, k = 500, 10, 4
    run = S.Run(S.Dataset.from_bits(X, hard), n, seed=7, chain_offset=1000, store=S.STORE_PI, max_samples=samp)
    run.init().advance_both(15, samp)
    res = run.cross_chain(k)
    e = run.chain_stats()["e_negloglik"]
    want = oracle_mod.choose_chains(e, k)
    assert [c - 1000 for c in res["chosen"]] == want             # GLOBAL ids out
    assert res["min"] == e.min() and abs(res["sigma"] - np.std(e)) < 1e-9
    assert np.array_equal(res["counts"], run.po_counts(np.array(want, np.int32) + 1000))
    for c, ch in enumerate(want):
        assert np.array_equal(res["counts"][c], oracle_mod.pair_order_counts(run.fetch_samples(ch, full=False)["pi"]))
    # a one-rank NCCL communicator goes through the collective code path and changes nothing
    comm = S.Comm(S.Comm.unique_id(), 1, 0, 0)
    run0 = S.Run(S.Dataset.from_bits(X, hard), n, seed=7, chain_offset=1000, store=S.STORE_PI, max_samples=samp).init().advance_both(15, samp)
    res0 = run0.cross_chain(k, comm=comm)
    assert [c - 1000 for c in res0["chosen"]] == want and np.array_equal(res0["counts"], res["counts"])
    comm.close()


def test_pair_order_uses_each_chains_own_sample_count(S, oracle_mod):
    """a chain whose tape ran out early holds fewer samples than chain 0: its slab counts ITS samples (round 1 took T
    from chain 0 for every chain)"""
    X, hard = load_hex_dataset("g10s10")
    full = _oracle_chain(oracle_mod, X, hard, 5, 0, 6)
    short = _oracle_chain(oracle_mod, X, hard, 6, 0, 3)
    run = S.Run(S.Dataset.from_bits(X, hard), 2, mode=S.MODE_REPLAY, store=S.STORE_PI, max_samples=6)
    run.set_tapes([full[4], short[4]]).init().advance(6, True).sync()
    counts = run.po_counts(np.array([0, 1], np.int32))
    assert counts[0][0, 0] == -6 and counts[1][0, 0] == -3
    assert np.array_equal(counts[1], oracle_mod.pair_order_counts(short[2]["pi"]))
    with pytest.raises(S.SeriationError):
        run.posterior_sums([0, 1])          # the mirrors assume one T: chains that disagree are refused, not mis-scaled


def test_site_age_correlation_against_numpy(S, tmp_path):
    """CORR_MN (Report Table 1) with the .sites chronology in place of the file order"""
    X, hard = load_hex_dataset("g10s10")
    N, M = X.shape
    rng = np.random.default_rng(5)
    mn = np.sort(rng.integers(2, 14, N))
    age = np.round(22.0 - 1.1 * mn + rng.random(N) * 0.5, 2)
    (tmp_path / "t.genus").write_text("".join("G%d \n" % m for m in range(M)))
    (tmp_path / "t.sites").write_text("".join("S%d [%d,%s]%s\n" % (n, mn[n], repr(float(age[n])), " *" if hard[n] else "") for n in range(N)))
    ds = S.Dataset.from_bits(X, hard).read_names(str(tmp_path / "t.genus"), str(tmp_path / "t.sites"))
    run = S.Run(ds, 40, seed=3, store=S.STORE_PI, max_samples=30).init().advance_both(100, 30).sync()
    chosen = S.select_chains(run.chain_stats()["e_negloglik"], 3)[0]
    ca, cm = run.site_age_corr(chosen)
    pis = [run.fetch_samples(int(c), full=False)["pi"] for c in chosen]
    want_mn = np.mean([np.mean([np.corrcoef(p, mn)[0, 1] for p in ps]) for ps in pis])
    want_age = np.mean([np.mean([np.corrcoef(p, -age)[0, 1] for p in ps]) for ps in pis])
    assert abs(cm - want_mn) < 1e-12 and abs(ca - want_age) < 1e-12
    assert abs(cm) > 0.5                     # the sampler recovers the chronology (either direction of time)


# ----------------------------------------------------------------------------- round 2: multi-GPU behind the C ABI
def test_multi_on_one_device_equals_a_plain_run(S, oracle_mod):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    n, k = 700, 3
    m = S.Multi(ds, n, 1, seed=11, chain_offset=50, store=S.STORE_PI, max_samples=5).init().advance(6, 5).sync()
    assert m.check() == 0 and m.layout() == dict(n_gpus=1, chains_per_gpu=[n], peer_stores=True)
    run = S.Run(ds, n, seed=11, chain_offset=50, store=S.STORE_PI, max_samples=5).init().advance_both(6, 5).sync()
    assert m.chain_stats()["e_negloglik"].tobytes() == run.chain_stats()["e_negloglik"].tobytes()
    a, b = m.cross_chain(k), run.cross_chain(k)
    assert list(a["chosen"]) == list(b["chosen"]) and np.array_equal(a["counts"], b["counts"])
    r, loc = m.locate(50 + 123)
    assert loc == 123 and np.array_equal(r.state(loc)["pi"], run.state(123)["pi"])
    m.close()


def _device_count():
    import torch
    return torch.cuda.device_count()


@pytest.mark.parametrize("nccl", [False, True])
def test_multi_gpu_sharding_is_invisible(S, monkeypatch, nccl):
    """the chains of one call over all GPUs of the box (ser_multi_*): same chosen chains, same pair-order counts, same
    per-chain statistics as one GPU, through the kernels' own peer stores and through NCCL"""
    G = _device_count()
    if G < 2:
        pytest.skip("one GPU on this box")
    if nccl:
        monkeypatch.setenv("SER_MULTI_NCCL", "1")
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    n, k = 64 * G if nccl else 64 * G + 3, 4       # uneven blocks are fine with peer stores
    m = S.Multi(ds, n, G, seed=21, store=S.STORE_PI, max_samples=6).init().advance(8, 6).sync()
    assert m.check() == 0 and m.layout()["peer_stores"] == (not nccl)
    run = S.Run(ds, n, seed=21, store=S.STORE_PI, max_samples=6).init().advance_both(8, 6).sync()
    assert m.chain_stats()["e_negloglik"].tobytes() == run.chain_stats()["e_negloglik"].tobytes()
    for _ in range(2):                               # twice: the second call reuses the peer buffers
        a, b = m.cross_chain(k), run.cross_chain(k)
        assert list(a["chosen"]) == list(b["chosen"]) and a["min"] == b["min"] and a["sigma"] == b["sigma"]
        assert np.array_equal(a["counts"], b["counts"])
    m.close()


def test_cli_multi_gpu_and_index_check(S, tmp_path):
    import subprocess
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    ds = tmp_path / "g10s10.txt"
    write_txt(str(ds), X, hard)
    exe = os.path.join(S.PKG_DIR, "mcmc")
    with open(ds) as f:   # an index without a Chains/chain_XX directory is refused up front (it used to run and write nothing)
        r = subprocess.run([exe, "100"], stdin=f, cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 1 and "0..99" in r.stderr
    G = min(_device_count(), 8)
    outs = []
    for g in sorted({1, G}):
        out = subprocess.run([exe, "--chains", "640", "--gpus", str(g), "--burn", "10", "--samples", "8", "--seed", "4", "--dataset", str(ds),
                              "--select", "3", "--po", str(tmp_path / ("po%d.csv" % g))], check=True, capture_output=True, text=True)
        assert "gpus %d" % g in out.stdout and "no chain files" not in out.stderr
        outs.append([ln for ln in out.stdout.split("\n") if ln.startswith(("selection", "E[c]"))])
        po = np.loadtxt(tmp_path / ("po%d.csv" % g), delimiter=",")
        assert po.shape == (124, 124)
    assert all(o == outs[0] for o in outs)
    if G > 1:
        assert (tmp_path / "po1.csv").read_bytes() == (tmp_path / ("po%d.csv" % G)).read_bytes()


# ----------------------------------------------------------------------------- round 2: per-taxon c, d for large shapes
@pytest.mark.parametrize("threads", ["64", "1024"])
def test_manycd_big_path_replay_bit_exact(S, oracle_mod, monkeypatch, threads):
    """manycd = 1 through the large-shape slot kernel (mcmc.c:777-785, :807-815 work for any M): replay vs the oracle after every
    call, incl. every per-taxon c, d and the saved log-likelihood bits"""
    monkeypatch.setenv("SER_FORCE_BIG", threads)
    for name, burn, samp in (("g10s10", 6, 6), ("g5s5", 2, 2)):
        X, hard = load_hex_dataset(name)
        _manycd_replay_case(S, oracle_mod, X, hard, [31, 0], burn, samp)
    rng = np.random.default_rng(11)
    for shape in EDGE_SHAPES[1::3]:
        X, hard = random_dataset(rng, *shape)
        _manycd_replay_case(S, oracle_mod, X, hard, [4], 5, 5)


def test_manycd_wide_matrix_replay_and_free_running(S, oracle_mod):
    """more taxa than a CTA has threads (200 x 1500): per-taxon c, d on the large-shape kernel, replay and free-running"""
    X, hard = S.Dataset.synthetic(200, 1500, 6, 11).arrays()
    _manycd_replay_case(S, oracle_mod, X, hard, [1, 2], 2, 2)
    seed, offset = 99, 5
    run = S.Run(S.Dataset.from_bits(X, hard), 3, mode=S.MODE_FREE, seed=seed, chain_offset=offset, manycd=True)
    run.init().advance(2, False).advance(2, True).sync()
    assert run.check() == 0
    for i in range(3):
        o = _manycd_oracle(oracle_mod, X, hard, philox=(seed, offset + i), detmath=True)
        for _ in range(4):
            o.sample()
        _cmp_manycd(run, i, o.state(), ("free", i), True)
    run.close()


# ----------------------------------------------------------------------------- round 2: shapes beyond 1024 sites / 4096 taxa
@pytest.mark.parametrize("shape", [(1500, 60, 5, .05), (2048, 150, 12, .03), (2047, 33, 0, .1)])
def test_more_than_1024_sites_replay(S, oracle_mod, shape):
    """N up to 2048 (64 words per column) through the one-thread-per-column kernel"""
    rng = np.random.default_rng(shape[0])
    X, hard = random_dataset(rng, *shape)
    _replay_case(S, oracle_mod, X, hard, [1, 2], 2, 2)


def test_large_shapes_beyond_round1_limits(S, oracle_mod, monkeypatch):
    """2048 sites x 1200 taxa and 48 sites x 8000 taxa through the large-shape kernel (scalar and per-taxon c, d)"""
    rng = np.random.default_rng(5)
    X, hard = random_dataset(rng, 2048, 1200, 9, .02)
    _replay_case(S, oracle_mod, X, hard, [3], 1, 1)
    X, hard = random_dataset(rng, 48, 8000, 4, .15)
    _replay_case(S, oracle_mod, X, hard, [4], 2, 2)
    _manycd_replay_case(S, oracle_mod, X, hard, [5], 1, 2)
