"""Rank-normalised split-R-hat, bulk-ESS and tail-ESS pooled over chosen chains (ser_run_rank_diagnostics, DESIGN.md 3.9).

A float64 NumPy / SciPy reference of the contract (rankdata, ndtri, numpy.quantile and Stan's ESS loop transcribed line for
line) is checked on the CPU against known answers, and its site path (ranks, folds and quantiles from a histogram) against its
generic path.  On the GPU the entry point is compared with it on sampler traces and on crafted stores injected through a
checkpoint: q05 and q95 bit for bit, the other fields within rtol 1e-9 wherever every decision of the reference's loop lies
farther than 1e-9 from its boundary."""
import os
import struct
import subprocess

import numpy as np
import pytest
from scipy.special import ndtri
from scipy.stats import rankdata

from conftest import load_hex_dataset, random_dataset

FIELDS = ("rhat_bulk", "rhat_fold", "ess_bulk", "ess_mean", "ess_q05", "ess_q95", "q05", "q95")
MARGIN = 1e-9
RTOL = 1e-9


# ----------------------------------------------------------------------------- the reference
def split(traces):
    """chains' traces [k][T] (ascending global id) -> the m = 2k sequences [m][n]: first and last n = T // 2 samples of each"""
    x = np.asarray(traces, np.float64)
    n = x.shape[1] // 2
    return np.stack([h for tr in x for h in (tr[:n], tr[tr.size - n:])])


def znorm(flat):
    S = flat.size
    return ndtri((rankdata(flat, method="average") - 0.375) / (S + 0.25))


def seq_moments(y):
    """per-sequence means and variances (divisor n - 1); a constant sequence has its value as mean and variance 0 exactly"""
    const = y.min(axis=1) == y.max(axis=1)
    mean = np.where(const, y[:, 0], y.mean(axis=1))
    var = np.where(const, 0.0, y.var(axis=1, ddof=1))
    return mean, var


def rhat_basic(y):
    m, n = y.shape
    mean, var = seq_moments(y)
    W = var.mean()
    Bn = 0.0 if mean.min() == mean.max() else np.var(mean, ddof=1)
    if W == 0:
        return np.inf if Bn > 0 else np.nan
    return np.sqrt(((n - 1) / n * W + Bn) / W)


def ess(y, decisions=None):
    """Stan's multi-chain ESS (ArviZ's _ess) on sequences y [m][n], as the contract transcribes it; the value of every decision the
    loop takes is appended to `decisions` (its distance from the boundary is |value|)"""
    m, n = y.shape
    dec = decisions if decisions is not None else []
    if np.all(y == y.flat[0]):
        return np.nan
    mean, _ = seq_moments(y)
    yc = y - mean[:, None]

    def acov_mean(tau):
        return np.mean([np.dot(yc[j, :n - tau], yc[j, tau:]) / n for j in range(m)])

    mean_var = acov_mean(0) * n / (n - 1)
    var_plus = mean_var * (n - 1) / n + (0.0 if mean.min() == mean.max() else np.var(mean, ddof=1))

    def rho_hat(tau):
        return 1 - (mean_var - acov_mean(tau)) / var_plus

    rho = np.zeros(n)
    rho[0] = 1
    even = 1.0
    odd = rho[1] = rho_hat(1)
    t = 1
    while t < n - 3:
        dec.append(even + odd)
        if not even + odd > 0:
            break
        even, odd = rho_hat(t + 1), rho_hat(t + 2)
        dec.append(even + odd)
        if even + odd >= 0:
            rho[t + 1] = even
            rho[t + 2] = odd
        t += 2
    max_t = t - 2
    dec.append(even)
    if even > 0:
        rho[max_t + 1] = even
    t = 1
    while t <= max_t - 2:
        dec.append((rho[t + 1] + rho[t + 2]) - (rho[t - 1] + rho[t]))
        if rho[t + 1] + rho[t + 2] > rho[t - 1] + rho[t]:
            rho[t + 1] = rho[t + 2] = (rho[t - 1] + rho[t]) / 2
        t += 2
    tau = max(-1 + 2 * np.sum(rho[:max_t + 1]) + rho[max_t + 1], 1 / np.log10(m * n))
    ess.max_t = max_t
    return m * n / tau


def fields(y, z=None, zf=None, quant=None):
    """the eight fields of draws y [m][n] and the decisions behind fields 0..5; z, z_fold and (q05, q95, median) may be given (the
    site path), else they come from rankdata on the pooled draws"""
    m, n = y.shape
    flat = y.ravel()
    if quant is None:
        quant = (np.quantile(flat, 0.05), np.quantile(flat, 0.95), np.median(flat))
    q05, q95, med = quant
    if z is None:
        z = znorm(flat).reshape(m, n)
        zf = znorm(np.abs(flat - med)).reshape(m, n)
    dec = []
    out = [rhat_basic(z), rhat_basic(zf), ess(z, dec), ess(y, dec), ess((y <= q05).astype(np.float64), dec),
           ess((y <= q95).astype(np.float64), dec), q05, q95]
    return np.array(out), dec


def site_tables(hist, S):
    """the site path: z[p], z_fold[p], (q05, q95, median) from the pooled position histogram of one site"""
    N = hist.size
    C = np.concatenate([[0], np.cumsum(hist)])
    assert C[-1] == S

    def xs(j):
        return float(np.searchsorted(C[1:], j, side="right"))

    def lerp(a, b, t):
        d = b - a
        return a + d * t if t < 0.5 else b - d * (1 - t)

    qs = []
    for p in (0.05, 0.95):
        h = (S - 1) * p
        j = np.floor(h)
        qs.append(lerp(xs(int(j)), xs(min(int(j) + 1, S - 1)), h - j))
    med = (xs(S // 2 - 1) + xs(S // 2)) * 0.5
    z = ndtri((C[:-1] + (hist + 1) * 0.5 - 0.375) / (S + 0.25))
    m0 = int(np.floor(med))
    half = med != m0
    p = np.arange(N)
    s = np.where(p <= m0, m0 - p, p - m0 - half)
    F = np.zeros(N, np.int64)
    for k in range(N):
        lo, hi = m0 - k, (m0 + 1 + k if half else m0 + k)
        F[k] = (hist[lo] if lo >= 0 else 0) + (hist[hi] if hi != lo and hi < N else 0)
    CF = np.concatenate([[0], np.cumsum(F)])
    zf = ndtri((CF[s] + (F[s] + 1) * 0.5 - 0.375) / (S + 0.25))
    return z, zf, (qs[0], qs[1], med)


def fields_site(y, N):
    """fields() through the site path: y [m][n] integer positions in [0, N)"""
    hist = np.bincount(y.ravel().astype(np.int64), minlength=N)
    z, zf, quant = site_tables(hist, y.size)
    yi = y.astype(np.int64)
    return fields(y, z[yi], zf[yi], quant)


def far(dec):
    return all(abs(v) > MARGIN for v in dec)


# ----------------------------------------------------------------------------- CPU: the reference against known answers
@pytest.mark.parametrize("T", [40, 41, 200, 201])
def test_site_path_equals_generic_path(T):
    rng = np.random.default_rng(T)
    N = 12
    for trial in range(20):
        k = int(rng.integers(1, 5))
        w = rng.random(N) ** 4                                  # heavy ties, some positions never used
        traces = rng.choice(N, size=(k, T), p=w / w.sum())
        y = split(traces)
        flat = y.ravel()
        z, zf, quant = site_tables(np.bincount(flat.astype(np.int64), minlength=N), flat.size)
        yi = y.astype(np.int64)
        med = np.median(flat)
        assert quant[0] == np.quantile(flat, 0.05) and quant[1] == np.quantile(flat, 0.95) and quant[2] == med
        assert np.allclose(z[yi].ravel(), znorm(flat), rtol=1e-15, atol=1e-15)
        assert np.allclose(zf[yi].ravel(), znorm(np.abs(flat - med)), rtol=1e-15, atol=1e-15)
        a, b = fields(y)[0], fields_site(y, N)[0]
        assert np.allclose(a, b, rtol=1e-12, atol=0, equal_nan=True)


def test_odd_T_leaves_out_the_middle_sample():
    tr = np.arange(7.0)[None, :]
    assert split(tr).tolist() == [[0, 1, 2], [4, 5, 6]]


def test_iid_normal_gives_ess_near_S():
    rng = np.random.default_rng(1)
    y = split(rng.standard_normal((4, 4000)))
    S = y.size
    e = fields(y)[0]
    assert 0.9 * S < e[2] < 1.1 * S and 0.9 * S < e[3] < 1.1 * S
    assert abs(e[0] - 1) < 0.01 and abs(e[1] - 1) < 0.01


@pytest.mark.parametrize("phi", [0.5, 0.9])
def test_ar1_gives_the_known_ess(phi):
    rng = np.random.default_rng(2)
    k, T = 4, 40000
    e = rng.standard_normal((k, T))
    x = np.empty((k, T))
    x[:, 0] = e[:, 0] / np.sqrt(1 - phi * phi)
    for t in range(1, T):
        x[:, t] = phi * x[:, t - 1] + e[:, t]
    y = split(x)
    want = y.size * (1 - phi) / (1 + phi)
    assert abs(ess(y) / want - 1) < 0.1 and abs(ess(znorm(y.ravel()).reshape(y.shape)) / want - 1) < 0.1


def test_fold_sees_a_difference_in_spread_that_bulk_does_not():
    rng = np.random.default_rng(3)
    x = rng.standard_normal((4, 2000)) * np.array([1, 1, 3, 3])[:, None]
    f = fields(split(x))[0]
    assert abs(f[0] - 1) < 0.01 and f[1] > 1.1


def test_constant_sequences_at_different_levels_give_infinite_rhat():
    y = np.repeat(np.arange(6.0), 10).reshape(6, 10)
    assert rhat_basic(y) == np.inf
    assert np.isnan(rhat_basic(np.ones((6, 10))))
    assert np.isnan(ess(np.ones((6, 10))))


# ----------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


def dev_exp(v):
    """exp as the device computes it (libdevice): numpy's exp may differ from it in the last bit, and q05 / q95 are compared
    bit for bit"""
    import torch
    return torch.exp(torch.as_tensor(np.asarray(v, np.float64), device="cuda")).cpu().numpy()


def quantity_traces(loglik, c, d, pi):
    """per chain ([T] loglik, c, d and [T][N] pi) the traces of every quantity: [k][3 + N][T]"""
    return np.stack([np.concatenate([[-ll, dev_exp(cc), dev_exp(dd)], p.T.astype(np.float64)])
                     for ll, cc, dd, p in zip(loglik, c, d, pi)])


def compare(got, traces, N, what=3, label=""):
    """got: Run.rank_diagnostics; traces [k][3 + N][T].  Returns (compared, skipped) quantity counts."""
    qs = ([0, 1, 2] if what & 1 else []) + (list(range(3, 3 + N)) if what & 2 else [])
    done = skipped = 0
    for q in qs:
        y = split(traces[:, q, :])
        want, dec = fields_site(y, N) if q >= 3 else fields(y)
        g = np.array([got[f][q] for f in FIELDS])
        assert g[6:].tobytes() == want[6:].tobytes(), (label, q, g[6:], want[6:])
        if not far(dec):
            skipped += 1
            continue
        assert np.allclose(g[:6], want[:6], rtol=RTOL, atol=0, equal_nan=True), (label, q, g[:6], want[:6])
        done += 1
    for q in set(range(3 + N)) - set(qs):
        assert all(np.isnan(got[f][q]) for f in FIELDS)
    return done, skipped


def _run_traces(run, chosen, N):
    ll, c, d, pi = [], [], [], []
    for g in sorted(chosen):
        s = run.fetch_samples(g)
        ll.append(s["loglik"]); c.append(s["c"]); d.append(s["d"]); pi.append(s["pi"])
    return quantity_traces(ll, c, d, pi)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["g10s10", "g2s2"])
@pytest.mark.parametrize("T", [200, 201])
def test_sampler_traces_against_the_reference(S, name, T):
    X, hard = load_hex_dataset(name)
    ds = S.Dataset.from_bits(X, hard)
    run = S.Run(ds, 4, seed=31 + T, store=S.STORE_FULL, max_samples=T).init().advance(T, True).sync()
    got = run.rank_diagnostics([3, 1, 0, 2])
    done, skipped = compare(got, _run_traces(run, range(4), ds.N), ds.N, label=(name, T))
    assert skipped <= 0.1 * (done + skipped), (done, skipped)
    run.close()


@pytest.mark.gpu
@pytest.mark.parametrize("big", [False, True], ids=["one-thread-per-taxon", "large-shape"])
def test_manycd_scalars_are_taxon_0(S, big):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    if big:
        os.environ["SER_FORCE_BIG"] = "256"
    try:
        run = S.Run(ds, 4, seed=5, manycd=True, store=S.STORE_FULL, max_samples=120).init().advance(120, True).sync()
    finally:
        os.environ.pop("SER_FORCE_BIG", None)
    assert (run.kernel_path() != 0) == big
    tr = []
    for g in range(4):
        s = run.fetch_samples(g)
        assert s["c"].tobytes() == s["c_all"][:, 0].tobytes()
        tr.append((s["loglik"], s["c_all"][:, 0], s["d_all"][:, 0], s["pi"]))
    got = run.rank_diagnostics(range(4))
    done, skipped = compare(got, quantity_traces(*zip(*tr)), ds.N, label=("manycd", big))
    assert skipped <= 0.1 * (done + skipped), (done, skipped)
    run.close()


# ----------------------------------------------------------------------------- GPU: crafted stores through a checkpoint
HEADER = 104
K = 4
N_CRAFT = 48
T_GROUPS = [4, 5, 62, 63, 64, 66, 126, 128, 130, 400, 401, 401, 63]    # the last two repeat 401 and 63 with another middle row


def _fnv(data):
    h = 0xcbf29ce484222325
    for (w,) in struct.iter_unpack("<Q", data):
        h = ((h ^ w) * 0x100000001b3) & 0xffffffffffffffff
    return h


def _layout(N, M, store, rows):
    """byte offsets of the parts of a checkpoint record (DESIGN.md 3.6) of a run without manycd or accumulators"""
    o, L = 168, {}
    for name, nbytes in (("cdl", 8 * 3 * rows), ("rpi", 2 * N), ("ab", 4 * M), ("spi", 2 * N * rows), ("sa", 2 * M * rows),
                         ("sb", 2 * M * rows)):
        L[name] = o
        o += nbytes
    L["size"] = (o + 7) // 8 * 8 + 8
    return L


def _craft_chain(rng, c, T, R):
    """R rows of pi (permutations) and cdl = (c, d, loglik) for chosen chain c of a group; rows past T are never read.  Sites:
    0 constant everywhere; 1 constant in chain 0 only; 2 chains in disjoint ranges; 3 equal location, spread x 8 in chains 2, 3;
    4 each half constant at its own level; 5 q95 at the maximum; 6 a slowly mixing walk; the rest fill the free positions."""
    N, n = N_CRAFT, T // 2
    half = np.where(np.arange(R) < n, 0, 1)                     # rows of the first half, then the middle row and the second half
    drive = np.zeros((R, 7), np.int64)
    drive[:, 0] = 0
    drive[:, 1] = 1 if c == 0 else rng.integers(1, 4, R)
    drive[:, 2] = 4 + 2 * c + rng.integers(0, 2, R)
    drive[:, 3] = 20 + (rng.integers(-8, 9, R) if c >= 2 else rng.integers(-1, 2, R))
    drive[:, 4] = 29 + 2 * c + half
    drive[:, 5] = 37 + (rng.random(R) < 0.3)
    walk = np.cumsum(rng.random(R) < 0.03) + rng.integers(0, 8)
    drive[:, 6] = 39 + np.abs((walk % 14) - 7)                  # reflecting walk over [39, 47)
    pi = np.empty((R, N), np.uint16)
    pi[:, :7] = drive
    for t in range(R):
        free = np.setdiff1d(np.arange(N), drive[t])
        pi[t, 7:] = rng.permutation(free)
    assert np.array_equal(np.sort(pi, axis=1), np.tile(np.arange(N), (R, 1)))
    cdl = np.empty((R, 3))
    cdl[:, 0] = np.where(rng.random(R) < 0.7, np.log(0.01), np.log(0.02))          # two-level scalars: heavy ties
    cdl[:, 1] = np.where(rng.random(R) < 0.5, np.log(0.3), np.log(0.6))
    cdl[:, 2] = np.where(rng.random(R) < 0.4, -1000.5, -1001.25)
    return pi, cdl


def _crafted_stores():
    rng = np.random.default_rng(77)
    R = max(T_GROUPS)
    stores = []
    for gi, T in enumerate(T_GROUPS):
        stores.append([(T,) + _craft_chain(rng, c, T, R) for c in range(K)])
    for a, b in ((10, 11), (3, 12)):                            # the same stores but for the middle row of an odd T
        assert T_GROUPS[a] == T_GROUPS[b] and T_GROUPS[a] % 2
        mid = T_GROUPS[a] // 2
        for c in range(K):
            T, pi, cdl = stores[a][c]
            pi2, cdl2 = pi.copy(), cdl.copy()
            pi2[mid] = pi[mid][::-1]
            cdl2[mid] = (-700.0, 0.0, -1e12)
            stores[b][c] = (T, pi2, cdl2)
    return stores, R


@pytest.fixture(scope="module")
def crafted(S, tmp_path_factory):
    """one run of len(T_GROUPS) groups of K chains; group g holds chains K g .. K g + K - 1 with T_GROUPS[g] samples each"""
    stores, R = _crafted_stores()
    X, hard = random_dataset(np.random.default_rng(5), N_CRAFT, 6, 0, .2)
    ds = S.Dataset.from_bits(X, hard)
    n = K * len(T_GROUPS)
    kw = dict(seed=11, store=S.STORE_FULL, max_samples=R)
    f = str(tmp_path_factory.mktemp("rank") / "ck")
    S.Run(ds, n, **kw).init().advance(R, True).save_checkpoint(f).close()
    data = bytearray(open(f, "rb").read())
    size = struct.unpack_from("<Q", data, 88)[0]
    L = _layout(ds.N, ds.M, S.STORE_FULL, R)
    assert L["size"] == size
    first = HEADER + (4 * n + 7) // 8 * 8 + 8
    for g, group in enumerate(stores):
        for c, (T, pi, cdl) in enumerate(group):
            off = first + (K * g + c) * size
            rec = bytearray(data[off:off + size])
            rec[L["spi"]:L["spi"] + pi.nbytes] = pi.tobytes()
            rec[L["cdl"]:L["cdl"] + cdl.nbytes] = cdl.tobytes()
            struct.pack_into("<i", rec, 156, T)
            struct.pack_into("<Q", rec, size - 8, _fnv(bytes(rec[:size - 8])))
            data[off:off + size] = rec
    open(f, "wb").write(bytes(data))
    run = S.Run(ds, n, **kw).load_checkpoint(f)
    yield run, stores
    run.close()


def _crafted_traces(group):
    return quantity_traces([cdl[:, 2] for _, _, cdl in group], [cdl[:, 0] for _, _, cdl in group],
                           [cdl[:, 1] for _, _, cdl in group], [pi for _, pi, _ in group])


@pytest.mark.gpu
def test_crafted_stores_against_the_reference(S, crafted):
    run, stores = crafted
    results = []
    for g, group in enumerate(stores):
        T = group[0][0]
        ids = list(range(K * g, K * g + K))
        got = run.rank_diagnostics(ids[::-1])
        tr = _crafted_traces(group)[:, :, :T]
        compare(got, tr, N_CRAFT, label=("crafted", g, T))
        results.append(got)
        # site 0 constant in every chain: no R-hat, no ESS
        assert all(np.isnan(got[f][3]) for f in FIELDS[:6]) and got["q05"][3] == got["q95"][3] == 0
        # site 1 constant in chain 0 only: defined
        assert np.isfinite(got["rhat_bulk"][4])
        # site 4: every half constant at its own level
        assert got["rhat_bulk"][7] == np.inf and got["rhat_fold"][7] == np.inf
        # site 5: q95 is the maximum, so its indicator is constant
        assert got["q95"][8] == split(tr[:, 8, :]).max() and np.isnan(got["ess_q95"][8])
        if T >= 62:                                             # two-level scalars
            assert all(np.isfinite(got["rhat_bulk"][q]) and np.isfinite(got["ess_bulk"][q]) for q in range(3))
        if T >= 126:
            assert got["rhat_bulk"][5] > 1.5                   # site 2: chains in disjoint ranges
        if T >= 400:
            assert got["rhat_bulk"][6] < 1.05 and got["rhat_fold"][6] > 1.1   # site 3: only the fold sees the spread
            ess(split(tr[:, 9, :]))
            assert ess.max_t > 96                               # site 6: the loop runs past three lag blocks
    for a, b in ((10, 11), (3, 12)):                            # an extreme middle sample changes nothing
        for f in FIELDS:
            assert results[a][f].tobytes() == results[b][f].tobytes(), (a, b, f)


@pytest.mark.gpu
def test_errors_leave_out_untouched(S, crafted):
    import ctypes as C
    run, _ = crafted
    L = S.lib()
    Q = 3 + N_CRAFT
    out = np.full((Q, 8), 1234.5)

    def call(chosen, what=3, h=run._h, o=out, k=None):
        ch = None if chosen is None else np.ascontiguousarray(chosen, np.int32)
        ptr = None if ch is None else ch.ctypes.data_as(C.POINTER(C.c_int32))
        return L.ser_run_rank_diagnostics(h, ptr, len(chosen) if k is None else k, what,
                                          None if o is None else o.ctypes.data_as(C.POINTER(C.c_double)))

    E_ARG, E_STATE = -1, -4
    assert call([0, 1], k=0) == E_ARG
    assert call(None, k=2) == E_ARG
    assert call([0, 1], o=None) == E_ARG
    assert call([0, 1], h=None) == E_ARG
    assert call([0, 1], what=0) == E_ARG and call([0, 1], what=4) == E_ARG
    assert call([0, -1]) == E_ARG and call([1, 0, 1]) == E_ARG and call([0, 10 ** 6]) == E_ARG
    assert call([0, 4]) == E_STATE                              # T = 4 and T = 5
    assert np.all(out == 1234.5)
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    out_g = np.full((3 + ds.N, 8), 1234.5)                      # out is [3 + N][8] of the run's own dataset
    pi_only = S.Run(ds, 2, seed=1, store=S.STORE_PI, max_samples=8).init().advance(8, True).sync()
    assert call([0, 1], h=pi_only._h, o=out_g) == E_STATE
    assert np.all(out_g == 1234.5)
    assert call([0, 1], what=2, h=pi_only._h, o=out_g) == 0 and np.all(out_g[:3] == 1234.5)
    out_g[:] = 1234.5
    none = S.Run(ds, 2, seed=1, store=S.STORE_NONE, max_samples=8).init().advance(8, True).sync()
    assert call([0, 1], what=2, h=none._h, o=out_g) == E_STATE
    fresh = S.Run(ds, 2, seed=1, store=S.STORE_FULL, max_samples=8)
    assert call([0, 1], h=fresh._h, o=out_g) == E_STATE
    short = S.Run(ds, 2, seed=1, store=S.STORE_FULL, max_samples=8).init().advance(3, True).sync()
    assert call([0, 1], h=short._h, o=out_g) == E_STATE
    acc = S.Run(ds, 2, seed=1, store=S.STORE_FULL, max_samples=8).init()
    acc.accumulate()
    acc.advance(8, True).sync()
    assert call([0, 1], h=acc._h, o=out_g) == E_STATE
    assert np.all(out_g == 1234.5) and np.all(out == 1234.5)
    with pytest.raises(S.SeriationError, match=r"^\[-1\]"):
        run.rank_diagnostics([2, 2])
    with pytest.raises(S.SeriationError, match=r"^\[-4\]"):
        run.rank_diagnostics([0, 4])
    # rows that are not requested keep what the caller passed
    assert call([0, 1, 2, 3], what=2) == 0
    assert np.all(out[:3] == 1234.5) and not np.any(out[3:] == 1234.5)
    out[:] = 1234.5
    assert call([0, 1, 2, 3], what=1) == 0
    assert np.all(out[3:] == 1234.5) and not np.any(out[:3] == 1234.5)
    for r in (pi_only, none, fresh, short, acc):
        r.close()


# ----------------------------------------------------------------------------- GPU: the same bits on any run that holds the chains
def _same(a, b, what):
    for f in a:
        assert a[f].tobytes() == b[f].tobytes(), (what, f)


@pytest.mark.gpu
def test_same_bits_on_any_run_holding_the_chains(S, tmp_path):
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    kw = dict(seed=9, store=S.STORE_FULL, max_samples=90)
    full = S.Run(ds, 8, **kw).init().advance(10, False).advance(90, True).sync()
    ids = [5, 2, 3, 4]
    want = full.rank_diagnostics(ids)
    _same(want, full.rank_diagnostics(sorted(ids)), "permuted chosen")
    sub = S.Run(ds, 4, chain_ids=np.array([4, 2, 5, 3], np.int32), **kw).init().advance(10, False).advance(90, True).sync()
    _same(want, sub.rank_diagnostics(ids), "subset run")
    shard = S.Run(ds, 4, chain_offset=2, **kw).init().advance(10, False).advance(90, True).sync()
    _same(want, shard.rank_diagnostics(ids), "sharded run")
    half = S.Run(ds, 8, **kw).init().advance(10, False).advance(40, True)
    f = str(tmp_path / "ck")
    half.save_checkpoint(f)
    half.close()
    resumed = S.Run(ds, 8, **kw).load_checkpoint(f).advance(50, True).sync()
    _same(want, resumed.rank_diagnostics(ids), "resumed run")
    for r in (full, sub, shard, resumed):
        r.close()


# ----------------------------------------------------------------------------- CLI
def test_cli_rank_diagnostics_needs_select(S, tmp_path):
    r = subprocess.run([os.path.join(S.PKG_DIR, "mcmc"), "--chains", "4", "--rank-diagnostics", str(tmp_path / "r.csv")],
                       capture_output=True, text=True)
    assert r.returncode == 1 and "--rank-diagnostics" in r.stderr and not (tmp_path / "r.csv").exists()


@pytest.mark.gpu
def test_cli_rank_diagnostics(S, tmp_path):
    from tools.datasets import write_txt
    X, hard = load_hex_dataset("g10s10")
    write_txt(str(tmp_path / "g10s10.txt"), X, hard)
    burn, samp = 20, 60
    base = [os.path.join(S.PKG_DIR, "mcmc"), "--chains", "64", "--burn", str(burn), "--samples", str(samp), "--seed", "0", "--select", "4",
            "--dataset", str(tmp_path / "g10s10.txt")]
    env = {k: v for k, v in os.environ.items() if k != "GSL_RNG_SEED"}
    run = lambda extra: subprocess.run(base + extra, check=True, capture_output=True, text=True, env=env).stdout.splitlines()
    out = run(["--rank-diagnostics", str(tmp_path / "r.csv")])
    line = [x for x in out if x.startswith("rank diagnostics:")]
    assert len(line) == 1 and "R-hat max" in line[0] and "tail-ESS min" in line[0]
    lines = open(tmp_path / "r.csv").read().splitlines()
    assert lines[0] == "quantity,rhat,rhat_bulk,rhat_fold,ess_bulk,ess_tail,ess_mean,q05,q95"
    N = X.shape[0]
    assert [ln.split(",")[0] for ln in lines[1:]] == ["-logL", "c", "d"] + ["site_%d" % i for i in range(N)]
    rows = np.array([[float(v) for v in ln.split(",")[1:]] for ln in lines[1:]])
    # the same chains in Python
    first = S.run_all_chains(S.Dataset.from_bits(X, hard), 64, burn, samp, seed=0, store=S.STORE_NONE)
    chosen = S.choose_chains(first, 4)
    assert ("chosen " + " ".join(map(str, chosen))) in [x for x in out if x.startswith("selection:")][0]
    rd = S.rank_diagnostics(S.replay_chosen(first, chosen, window=0), chosen)
    want = np.column_stack([rd[f] for f in ("rhat", "rhat_bulk", "rhat_fold", "ess_bulk", "ess_tail", "ess_mean", "q05", "q95")])
    assert rows.shape == (3 + N, 8) and np.array_equal(rows, want, equal_nan=True)
    flagged = sum(1 for r in rows if r[0] > 1.01 or r[3] < 400 or r[4] < 400)
    assert line[0].endswith("%d of %d quantities with R-hat > 1.01 or ESS < 400" % (flagged, 3 + N))
    # with --diagnostics too: one replay, and the --diagnostics file does not change
    run(["--diagnostics", str(tmp_path / "d1.csv")])
    both = run(["--diagnostics", str(tmp_path / "d2.csv"), "--rank-diagnostics", str(tmp_path / "r2.csv")])
    assert (tmp_path / "d2.csv").read_bytes() == (tmp_path / "d1.csv").read_bytes()
    assert (tmp_path / "r2.csv").read_bytes() == (tmp_path / "r.csv").read_bytes()
    assert len([x for x in both if x.startswith("diagnostics:")]) == 1
