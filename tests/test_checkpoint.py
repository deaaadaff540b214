"""Checkpoint and resume: every chain of a run saved to a file and continued in another run, bit for bit, on every sweep path,
in replay mode, with accumulating summaries, across shardings, and through the `mcmc` CLI; and the refusals of a file that
does not fit the run, which must never reach a sweep kernel."""
import ctypes as C
import os
import struct
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, load_hex_dataset

E_ARG, E_STATE, E_IO, E_TAPE, E_CHECK = -1, -4, -5, -6, -7
HEADER = 104


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


# ----------------------------------------------------------------------------- the format, as DESIGN.md section 3.6 states it
def _fnv(data: bytes) -> int:
    """FNV-1a over little-endian 64-bit words"""
    h = 0xcbf29ce484222325
    for (w,) in struct.iter_unpack("<Q", data):
        h = ((h ^ w) * 0x100000001b3) & 0xffffffffffffffff
    return h


def _layout(N, M, manycd, store, rows, acc):
    """byte offsets of a record's parts and its size"""
    o, L, full = 168, {}, store >= 2

    def take(name, nbytes):
        nonlocal o
        L[name] = o
        o += nbytes
    take("cd", 8 * 4 * M if manycd else 0)
    take("cdl", 8 * 3 * rows if full else 0)
    take("cd_all", 8 * 2 * M * rows if full and manycd else 0)
    take("po", 4 * N * N if acc & 1 else 0)
    take("pi", 4 * N if acc & 6 else 0)
    take("asum", 4 * M if acc & 4 else 0)
    take("bsum", 4 * M if acc & 4 else 0)
    take("alive", 4 * N * M if acc & 8 else 0)
    take("pos", 4 * N * N if acc & 16 else 0)
    take("range", 8 * M * (N + 1) if acc & 32 else 0)
    take("rpi", 2 * N)
    take("ab", 4 * M)
    take("spi", 2 * N * rows if store >= 1 else 0)
    take("sa", 2 * M * rows if full else 0)
    take("sb", 2 * M * rows if full else 0)
    L["size"] = (o + 7) // 8 * 8 + 8
    return L


def _header(N, M, n_chains, calls, n_samples, seed=7, mode=0, manycd=0, store=0, max_samples=0, acc=0):
    rows = max(0, min(n_samples, max_samples)) if store else 0
    size = _layout(N, M, manycd, store, rows, acc)["size"]
    body = b"SERCKPT\0" + struct.pack("<IIiiiiQIiiiiiqiiiiQ", 1, HEADER, N, M, 0, mode, 0x1234, seed, 10, manycd, store, max_samples, acc,
                                      calls, n_samples, 0, rows, n_chains, size)
    return body + struct.pack("<Q", _fnv(body)), size


def _file(N, M, ids, calls, n_samples, **kw):
    head, size = _header(N, M, len(ids), calls, n_samples, **kw)
    table = struct.pack("<%di" % len(ids), *ids)
    table += b"\0" * (-len(table) % 8)
    return head + table + struct.pack("<Q", _fnv(table)) + b"\0" * (size * len(ids))


def _info(S, path):
    return S.checkpoint_info(str(path))


# ----------------------------------------------------------------------------- host only
def test_checkpoint_info_reads_a_header_without_cuda(S, tmp_path):
    f = tmp_path / "ck"
    f.write_bytes(_file(9, 5, [0, 3, 8], 27, 7, seed=123, manycd=1))
    assert _info(S, f) == dict(N=9, M=5, n_chains=3, calls_done=27, n_samples=7, seed=123, mode=0, manycd=True)


def test_checkpoint_info_refuses_damaged_files(S, tmp_path):
    good = _file(9, 5, [0, 1], 4, 0)
    cases = {"missing": None, "truncated": good[:-1], "extended": good + b"\0" * 8, "magic": b"XERCKPT\0" + good[8:],
             "header checksum": good[:20] + bytes([good[20] ^ 1]) + good[21:]}
    for what, data in cases.items():
        f = tmp_path / what.replace(" ", "_")
        if data is not None:
            f.write_bytes(data)
        _raises(S, E_IO, _info, S, f)
    assert "bad magic" in _raises(S, E_IO, _info, S, tmp_path / "magic")
    assert "header checksum" in _raises(S, E_IO, _info, S, tmp_path / "header_checksum")


def test_cli_checkpoint_flags_need_a_checkpoint_file(S):
    exe = os.path.join(S.PKG_DIR, "mcmc")
    for extra in (["--stop-after", "3"], ["--checkpoint-every", "2"], ["--resume"]):
        r = subprocess.run([exe, "--chains", "4"] + extra, capture_output=True, text=True, stdin=subprocess.DEVNULL)
        assert r.returncode == 1 and "usage:" in r.stderr and "--checkpoint FILE" in r.stderr, extra


# ----------------------------------------------------------------------------- GPU
PATHS = {"default": {}, "big_groups": {"SER_FORCE_BIG": "256", "SER_BIG_WARP": "0"},
         "big_warp": {"SER_FORCE_BIG": "256", "SER_BIG_WARP": "1"}, "manycd": {}}


def _advance(run, done, n, burn):
    """calls [done, done + n) of a schedule whose first `burn` calls are burn-in"""
    b = max(0, min(n, burn - done))
    return run.advance_both(b, n - b)


def _same_chain(x, cx, y, cy, many, tmp_path=None):
    for k, v in x.state(cx).items():
        assert np.array_equal(v, y.state(cy)[k]), k
    assert np.array_equal(x.counters(cx), y.counters(cy))
    for k, v in x.fetch_samples(cx).items():
        assert np.array_equal(v, y.fetch_samples(cy)[k]), ("samples", k)
    if many:
        assert np.stack(x.cd(cx)).tobytes() == np.stack(y.cd(cy)).tobytes()
    if tmp_path is not None:
        for d, r, c in (("x", x, cx), ("y", y, cy)):
            (tmp_path / d).mkdir(parents=True, exist_ok=True)
            r.write_chain_files(c, str(tmp_path / d))
        files = sorted(os.listdir(tmp_path / "x"))
        assert len(files) == 5 and sorted(os.listdir(tmp_path / "y")) == files
        for f in files:
            assert (tmp_path / "x" / f).read_bytes() == (tmp_path / "y" / f).read_bytes(), f


def _same_stats(x, y):
    a, b = x.chain_stats(), y.chain_stats()
    assert a["n_samples"] == b["n_samples"]
    for k in ("e_negloglik", "e_c", "e_d"):
        assert a[k].tobytes() == b[k].tobytes(), k


@pytest.mark.gpu
@pytest.mark.parametrize("name,path", [("g10s10", p) for p in PATHS] + [("g2s2", "default")])
def test_split_run_equals_the_run_in_one_piece(S, monkeypatch, tmp_path, name, path):
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)
    ds = S.Dataset.from_bits(*load_hex_dataset(name))
    n, burn, samp, many = 12, 6, 5, path == "manycd"
    kw = dict(seed=21, store=S.STORE_FULL, max_samples=samp, manycd=many)
    whole = S.Run(ds, n, **kw).init().advance_both(burn, samp).sync()
    for split in (3, burn, 8):                                  # mid burn-in, the burn/sample boundary, mid sampling
        f = tmp_path / ("ck%d" % split)
        first = _advance(S.Run(ds, n, **kw).init(), 0, split, burn).save_checkpoint(f)
        assert _info(S, f)["calls_done"] == split and _info(S, f)["n_samples"] == max(0, split - burn)
        first.close()
        second = S.Run(ds, n, **kw).load_checkpoint(f)
        _advance(second, split, burn + samp - split, burn).sync()
        assert second.check() == 0
        _same_stats(second, whole)
        for c in range(n):
            _same_chain(second, c, whole, c, many, tmp_path / ("files%d" % split) if c == 1 else None)
        second.close()


@pytest.mark.gpu
def test_replay_run_resumes_mid_tape(S):
    g = np.load(os.path.join(GOLDEN, "ref_g10s10.npz"))
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    calls = len(g["kind"]) - 1
    kw = dict(mode=S.MODE_REPLAY, store=S.STORE_FULL, max_samples=calls)
    whole = S.Run(ds, 1, **kw).set_tapes([g["tape"]]).init().advance(calls, True).sync()
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        f = os.path.join(d, "ck")
        S.Run(ds, 1, **kw).set_tapes([g["tape"]]).init().advance(calls // 2, True).save_checkpoint(f)
        assert _info(S, f)["mode"] == S.MODE_REPLAY
        # tapes come first; a tape shorter than the saved cursor is refused before any sweep
        _raises(S, E_TAPE, S.Run(ds, 1, **kw).load_checkpoint, f)
        short = S.Run(ds, 1, **kw).set_tapes([g["tape"][:10]])
        assert "beyond its tape" in _raises(S, E_TAPE, short.load_checkpoint, f)
        _raises(S, E_STATE, short.advance, 1, True)
        rest = S.Run(ds, 1, **kw).set_tapes([g["tape"]]).load_checkpoint(f).advance(calls - calls // 2, True).sync()
    a, b = rest.state(0), whole.state(0)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert a["slots"] == int(g["slots"][-1]) == g["tape"].size
    for k in ("a", "b", "pi"):
        assert np.array_equal(a[k], g[k][-1].astype(np.int32)), k
    assert a["loglik"] == g["cdl"][-1][2]
    fa, fb = rest.fetch_samples(0), whole.fetch_samples(0)
    for k in fa:
        assert fa[k].tobytes() == fb[k].tobytes(), k
    assert np.array_equal(fa["loglik"], g["cdl"][1:, 2])
    _same_stats(rest, whole)


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


@pytest.mark.gpu
def test_accumulating_run_resumes_mid_window(S, tmp_path):
    ds = _dataset_with_ages(S, tmp_path)
    burn, T, chosen, kw = 5, 50, np.array([1, 4, 5], np.int32), dict(seed=4, store=S.STORE_FULL, max_samples=16)
    whole = S.Run(ds, 6, **kw).init().accumulate(ab=True, alive=True).advance(burn, False).advance(T, True).sync()
    f = tmp_path / "ck"
    S.Run(ds, 6, **kw).init().accumulate(ab=True, alive=True).advance(burn, False).advance(23, True).save_checkpoint(f)
    _raises(S, E_STATE, S.Run(ds, 6, **kw).load_checkpoint, f)          # the accumulators come first
    rest = S.Run(ds, 6, **kw).accumulate(ab=True, alive=True).load_checkpoint(f).advance(T - 23, True).sync()
    want, got = _summaries(whole, chosen), _summaries(rest, chosen)
    assert want["t"] == T
    for k in want:
        assert np.array_equal(np.asarray(got[k]), np.asarray(want[k])), k
    _same_stats(rest, whole)


@pytest.mark.gpu
def test_accumulator_parts_sit_where_the_layout_puts_them(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    N, M, n, T = ds.N, ds.M, 3, 23
    flags = dict(po=True, sums=True, ab=True, alive=True, positions=True, ranges=True)
    run = S.Run(ds, n, seed=9, store=S.STORE_FULL, max_samples=16).init().accumulate(**flags).advance(4, False).advance(T, True).sync()
    f = tmp_path / "ck"
    run.save_checkpoint(f)                                              # mid-window: 23 samples through a window of 16
    data = f.read_bytes()
    acc, rows, size = struct.unpack_from("<i", data, 60)[0], struct.unpack_from("<i", data, 80)[0], struct.unpack_from("<Q", data, 88)[0]
    assert acc == 63
    L = _layout(N, M, 0, S.STORE_FULL, rows, acc)
    assert L["size"] == size
    chosen = list(range(n))
    po, ps, (alive, t), m = run.po_counts(chosen), run.posterior_sums(chosen, with_ab=True), run.alive_counts(chosen), run.marginals(chosen, ranges=True)
    assert t == ps["n_samples"] == T
    first = HEADER + (4 * n + 7) // 8 * 8 + 8
    for c in range(n):
        rec = data[first + c * size:first + (c + 1) * size]

        def part(name, *shape):
            return np.frombuffer(rec, np.int32, int(np.prod(shape)), L[name]).reshape(shape)
        want_po = po[c].copy()
        np.fill_diagonal(want_po, 0)
        assert np.array_equal(part("po", N, N), want_po), c
        assert np.array_equal(part("pi", N), ps["pi_sum"][c]), c
        assert np.array_equal(part("asum", M), ps["a_sum"][c]) and np.array_equal(part("bsum", M), ps["b_sum"][c]), c
        assert np.array_equal(np.cumsum(part("alive", N, M), axis=0), alive[c]), c
        assert np.array_equal(part("pos", N, N), m["pos"][c]), c
        ab = part("range", 2, M, N + 1)
        assert np.array_equal(ab[0], m["a"][c]) and np.array_equal(ab[1], m["b"][c]), c


@pytest.mark.gpu
def test_a_subset_run_reads_its_own_chains(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    kw, f = dict(seed=8, store=S.STORE_FULL, max_samples=5), tmp_path / "ck"
    full = S.Run(ds, 40, **kw).init().advance(3, False).advance(2, True).save_checkpoint(f).advance(3, True).sync()
    ids = [31, 2, 17]
    sub = S.Run(ds, 0, chain_ids=ids, **kw).load_checkpoint(f).advance(3, True).sync()
    for c, g in enumerate(ids):
        _same_chain(sub, c, full, g, False)
    assert sub.chain_stats()["e_negloglik"].tobytes() == full.chain_stats()["e_negloglik"][ids].tobytes()
    assert "chain 40 is not in" in _raises(S, E_ARG, S.Run(ds, 0, chain_ids=[3, 40], **kw).load_checkpoint, f)


def _n_devices():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
def test_the_same_chains_give_the_same_bytes_whatever_the_sharding_or_path(S, monkeypatch, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, kw = 24, dict(seed=5, store=S.STORE_PI, max_samples=4)
    files = {}
    files["run"] = S.Run(ds, n, **kw).init().advance_both(4, 3).save_checkpoint(tmp_path / "run")
    files["permuted subset"] = S.Run(ds, 0, chain_ids=list(range(n))[::-1], **kw).init().advance_both(4, 3).save_checkpoint(tmp_path / "perm")
    files["multi1"] = S.Multi(ds, n, 1, **kw).init().advance(4, 3).save_checkpoint(tmp_path / "multi1")
    if _n_devices() >= 2:
        files["multi2"] = S.Multi(ds, n, 2, **kw).init().advance(4, 3).save_checkpoint(tmp_path / "multi2")
    monkeypatch.setenv("SER_FORCE_BIG", "256")
    big = S.Run(ds, n, **kw).init()
    assert big.kernel_path() != 0
    files["large-shape kernel"] = big.advance(4, False).advance(3, True).save_checkpoint(tmp_path / "big")
    names = {"run": "run", "permuted subset": "perm", "multi1": "multi1", "multi2": "multi2", "large-shape kernel": "big"}
    ref = (tmp_path / "run").read_bytes()
    for k in files:
        assert (tmp_path / names[k]).read_bytes() == ref, k
    assert len(ref) == HEADER + (n * 4 + 8) + n * _layout(ds.N, ds.M, 0, 1, 3, 0)["size"]


@pytest.mark.gpu
def test_multi_and_run_files_load_into_each_other(S, tmp_path):
    if _n_devices() < 2:
        pytest.skip("needs two devices")
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    n, kw = 20, dict(seed=6, store=S.STORE_PI, max_samples=6)
    whole = S.Run(ds, n, **kw).init().advance_both(3, 6).sync()
    S.Multi(ds, n, 2, **kw).init().advance(3, 2).save_checkpoint(tmp_path / "m")
    one = S.Run(ds, n, **kw).load_checkpoint(tmp_path / "m").advance_both(0, 4).sync()
    S.Run(ds, n, **kw).init().advance_both(3, 2).save_checkpoint(tmp_path / "r")
    two = S.Multi(ds, n, 2, **kw).load_checkpoint(tmp_path / "r").advance(0, 4).sync()
    assert one.chain_stats()["e_negloglik"].tobytes() == whole.chain_stats()["e_negloglik"].tobytes()
    assert two.chain_stats()["e_negloglik"].tobytes() == whole.chain_stats()["e_negloglik"].tobytes()
    assert two.cross_chain(3)["counts"].tobytes() == whole.cross_chain(3)["counts"].tobytes()
    for g in (0, 13, 19):
        r, c = two.locate(g)
        _same_chain(r, c, whole, g, False)
        _same_chain(one, g, whole, g, False)


def _patch_record(path, chain_pos, edit):
    """apply edit(record bytearray, layout) to one record and recompute its checksum"""
    data = bytearray(open(path, "rb").read())
    N, M, n_chains = struct.unpack_from("<ii", data, 16) + (struct.unpack_from("<i", data, 84)[0],)
    manycd, store, max_samples, acc = struct.unpack_from("<iiii", data, 48)
    rows, size = struct.unpack_from("<i", data, 80)[0], struct.unpack_from("<Q", data, 88)[0]
    L = _layout(N, M, manycd, store, rows, acc)
    assert L["size"] == size
    off = HEADER + (4 * n_chains + 7) // 8 * 8 + 8 + chain_pos * size
    rec = bytearray(data[off:off + size])
    edit(rec, L)
    struct.pack_into("<Q", rec, size - 8, _fnv(bytes(rec[:size - 8])))
    data[off:off + size] = rec
    return bytes(data)


@pytest.mark.gpu
def test_refusals_leave_the_run_unusable_and_sweep_nothing(S, tmp_path):
    X, hard = load_hex_dataset("g10s10")
    ds = S.Dataset.from_bits(X, hard)
    base = dict(seed=3, store=S.STORE_FULL, max_samples=4, sweeps_per_call=10)
    f = str(tmp_path / "ck")
    S.Run(ds, 4, **base).init().advance(2, False).advance(2, True).save_checkpoint(f)
    X2 = X.copy()
    X2[0, 0] ^= 1
    other = S.Dataset.from_bits(X2, hard)

    def refused(code, run, path=f, text=None):
        run.sweep_time(reset=True)
        msg = _raises(S, code, run.load_checkpoint, path)
        if text:
            assert text in msg, msg
        _raises(S, E_STATE, run.advance, 1, True)
        assert run.sweep_time()[1] == 0                               # no sweep launch since the load began
        return msg

    refused(E_ARG, S.Run(other, 4, **base), text="another dataset")
    refused(E_ARG, S.Run(S.Dataset.from_bits(*load_hex_dataset("g10s2")), 4, **base), text="another dataset")
    for field, change in (("seed", dict(seed=4)), ("mode", dict(mode=S.MODE_REPLAY)), ("manycd", dict(manycd=True)),
                          ("sweeps_per_call", dict(sweeps_per_call=9)), ("store", dict(store=S.STORE_PI)), ("max_samples", dict(max_samples=5))):
        refused(E_STATE, S.Run(ds, 4, **dict(base, **change)), text=field)
    refused(E_STATE, S.Run(ds, 4, **base).accumulate(), text="accumulate flags")
    refused(E_ARG, S.Run(ds, 0, chain_ids=[1, 7], **base), text="chain 7")
    # an initialised run that refuses a file is no longer initialised either
    refused(E_STATE, S.Run(ds, 4, **dict(base, seed=9)).init().advance(1, False))

    good = open(f, "rb").read()
    rs = struct.unpack_from("<Q", good, 88)[0]
    damaged = {"flip": good[:-rs // 2] + bytes([good[-rs // 2] ^ 0x40]) + good[-rs // 2 + 1:], "truncated": good[:-3]}
    for name, data in damaged.items():
        open(f + name, "wb").write(data)
        refused(E_IO, S.Run(ds, 4, **base), f + name)
    assert "checksum" in refused(E_IO, S.Run(ds, 4, **base), f + "flip")

    def dup_rpi(rec, L):
        rec[L["rpi"]:L["rpi"] + 2] = rec[L["rpi"] + 2:L["rpi"] + 4]

    def a_after_b(rec, L):
        M = ds.M
        struct.pack_into("<H", rec, L["ab"], 7)
        struct.pack_into("<H", rec, L["ab"] + 2 * M, 3)

    def loglik(rec, L):                                               # in range, but the totals no longer match: ser_check_kernel
        struct.pack_into("<d", rec, 32, struct.unpack_from("<d", rec, 32)[0] + 1.0)

    def stored_pi(rec, L):                                            # the histogram kernels index their rows with these
        struct.pack_into("<H", rec, L["spi"] + 2 * (ds.N + 3), ds.N)

    def stored_b(rec, L):
        struct.pack_into("<H", rec, L["sb"] + 2 * (ds.M + 5), ds.N + 1)

    for name, edit, text in (("pi", dup_rpi, "not a permutation"), ("ab", a_after_b, "a = 7, b = 3"), ("ll", loglik, "consistency check"),
                             ("spi", stored_pi, "stored row 1: spi is not a permutation"), ("sb", stored_b, "stored row 1: sa/sb of taxon 5")):
        open(f + name, "wb").write(_patch_record(f, 2, edit))
        refused(E_CHECK, S.Run(ds, 4, **base), f + name, text)
    refused(E_IO, S.Run(ds, 4, **base), str(tmp_path / "missing"))
    # the untouched file still loads and continues
    assert S.Run(ds, 4, **base).load_checkpoint(f).advance(2, True).sync().check() == 0


def _mcmc(S, cwd, *args):
    from tools.datasets import write_txt
    os.makedirs(cwd, exist_ok=True)
    txt = os.path.join(os.path.dirname(cwd), "g10s10.txt")
    if not os.path.exists(txt):
        write_txt(txt, *load_hex_dataset("g10s10"))
    cmd = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "12", "--burn", "20", "--samples", "10", "--select", "3", "--po", "po.csv",
           "--dataset", txt] + list(args)
    return subprocess.run(cmd, cwd=cwd, check=True, capture_output=True, text=True).stdout.splitlines()


def _untimed(lines, layout=True):
    """stdout without the timing fields of the first line (without that line when the device layout differs)"""
    return [x.split("  gpu_ms")[0] if x.startswith("chains ") else x for x in lines if layout or not x.startswith("chains ")]


def _tree(d):
    out = {}
    for root, _, files in os.walk(d):
        for f in files:
            p = os.path.join(root, f)
            out[os.path.relpath(p, d)] = open(p, "rb").read()
    return out


@pytest.mark.gpu
def test_cli_stop_and_resume_equal_the_one_shot_run(S, tmp_path):
    ref = _mcmc(S, str(tmp_path / "ref"))
    want_files = _tree(tmp_path / "ref")
    assert "po.csv" in want_files and sum(k.startswith("Chains") for k in want_files) == 12 * 5
    runs = [("split", [], [])]
    if _n_devices() >= 2:
        runs.append(("split2", ["--gpus", "2"], ["--gpus", "2"]))
    for name, first, second in runs:
        d = str(tmp_path / name)
        stop = _mcmc(S, d, "--checkpoint", "ck", "--stop-after", "13", *first)
        assert len(stop) == 1 and stop[0].startswith("stopped after call 13 of 30"), stop
        assert not os.path.exists(os.path.join(d, "Chains")) and not os.path.exists(os.path.join(d, "po.csv"))
        assert _info(S, os.path.join(d, "ck"))["calls_done"] == 13
        got = _mcmc(S, d, "--checkpoint", "ck", "--resume", *second)
        assert _untimed(got, not first) == _untimed(ref, not first), name
        files = _tree(d)
        files.pop("ck")
        assert files == want_files, name
    d = str(tmp_path / "every")
    got = _mcmc(S, d, "--checkpoint", "ck", "--checkpoint-every", "7")
    assert _untimed(got) == _untimed(ref)
    assert _info(S, os.path.join(d, "ck"))["calls_done"] == 30
    files = _tree(d)
    files.pop("ck")
    assert files == want_files
