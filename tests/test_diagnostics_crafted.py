"""ser_diag_kernel (DESIGN.md 3.7) against an exact reference on crafted traces injected through a checkpoint.

Every trace is x_t = base + scale * j_t with integer j_t, so the mean, the variances, every autocovariance and every Geyer pair
sum are exact rationals (mpmath at 256 bits for base and scale, Python ints for the sums over j).  The kernel is compared
with them under a forward-error bound derived from its summation orders (Higham's gamma_n), the error of its centring mean
and, for exp(c) and exp(d), one ulp on each input.  Every discrete decision -- a constant trace or half, each pair's P > 0,
gamma_0 >= DBL_MIN, the ESS floor -- is asserted exactly, after checking that the crafted trace keeps it farther from its
boundary than the bound.  The stores cover sample counts on both sides of the 32-lag block, the 64-sample chunk and the
96-sample sB window, tiles of Q = 32, 33, 64, 65 and 129 quantities, every `what`, max_lag at the block edges and at T,
chosen lists with repeats and ids the run does not hold, and split-R-hat over chains of equal T."""
import functools
import os
import struct
from fractions import Fraction

import mpmath
import numpy as np
import pytest

from conftest import random_dataset
from test_checkpoint import _layout, _patch_record
from test_diagnostics import ar1, ref_stats

mpmath.mp.prec = 256
mpf = mpmath.mpf
U = 2.0 ** -53                  # unit roundoff of float64
TINY = 2.0 ** -1074             # smallest subnormal: the absolute error of an underflowing product or quotient is below it
DBL_MIN = 2.0 ** -1022
SLACK = 1 + 2.0 ** -20          # covers the float64 evaluation of the bounds themselves


def gamma(n):
    return n * U / (1 - n * U)


def F(x):
    """a Fraction as an mpf (256 bits)"""
    return mpf(x.numerator) / x.denominator


# ----------------------------------------------------------------------------- the exact reference
class Trace:
    """x_t = base + scale * j_t exactly; the device reads values within `delta` of each x_t, equal j giving equal values
    (delta = 0 for integers and dyadic doubles, one ulp for exp).  With delta > 0 only two levels are allowed: the device
    trace is then again affine in j and has exactly the autocorrelations of j."""

    def __init__(self, j, base=0, scale=1, delta=0.0):
        self.j = np.asarray(j, np.int64)
        self.T = T = self.j.size
        self.base, self.scale, self.delta = mpf(base), mpf(scale), float(delta)
        assert delta == 0 or np.unique(self.j).size <= 2
        assert int(np.abs(self.j).max()) ** 2 * T < 2 ** 62          # the int64 lag products are exact
        self.S = int(self.j.sum())
        self.pre = np.concatenate([[0], np.cumsum(self.j)])
        self.G = []        # T^2 * sum_{t<T-k} (j_t - mu)(j_{t+k} - mu), exact
        self.E = []        # the kernel's error bound on sum_{t<T-k} (j_t - mu)(j_{t+k} - mu)
        self.geyer = None
        self.az = np.abs(self.j - self.S / T)
        self.xmax = max(abs(self.value(int(self.j.min()))), abs(self.value(int(self.j.max())))) + delta

    def value(self, j):
        return self.base + self.scale * (F(j) if isinstance(j, Fraction) else j)

    @functools.cached_property
    def moments(self):
        """(mean, e, var, e, constant) of the whole trace and of its two halves"""
        T, n = self.T, self.T // 2
        return _moments(self, 0, T), _moments(self, 0, n), _moments(self, T - n, T)

    def D(self, k):
        """|sum_{t<T-k} (j_t - mu)| + |sum_{t>=k} (j_t - mu)|: what a centring error e adds to lag k's sum, over e"""
        T, S = self.T, self.S
        return (abs(T * int(self.pre[T - k]) - (T - k) * S) + abs(T * (S - int(self.pre[k])) - (T - k) * S)) / T

    def G2(self, k):
        T, S = self.T, self.S
        while len(self.G) <= k:
            i = len(self.G)
            C = int(np.dot(self.j[:T - i], self.j[i:]))
            self.G.append(T * T * C - T * S * (int(self.pre[T - i]) + S - int(self.pre[i])) + (T - i) * S * S)
        return self.G[k]


def _mean_err(xmax, m, T):
    """|fl(sum x / count) - sum x / count| for pass 1's order: warp w sums t = w, w + 32, ... and one thread the 32 partials"""
    d = -(-T // 32) + 32
    return (gamma(d) * xmax * (1 + U) + U * abs(float(m)) + TINY) * SLACK


def _kernel_sum(x, lo, hi):
    """pass 1's sum over t in [lo, hi), in float64 and in its order: warp t mod 32 adds its samples in t order, then one
    thread adds the 32 partials in warp order (cumsum is sequential)"""
    t = np.arange(lo, hi)
    parts = np.array([x[t[t % 32 == w]].cumsum()[-1] if np.any(t % 32 == w) else 0.0 for w in range(32)])
    return parts.cumsum()[-1]


def _moments(tr, lo, hi):
    """mean and variance (divisor count - 1) of x over [lo, hi) with the kernel's error bounds, whether the part is constant,
    and a bound on the error of the device's centring mean.  With exact inputs that error is known: pass 1's sum is replayed
    in its order, and the device's mean must be that double."""
    j, T = tr.j[lo:hi], tr.T
    cnt = hi - lo
    if j.min() == j.max():
        return tr.value(int(j[0])), tr.delta, mpf(0), 0.0, True, 0.0, None
    S, SS = int(j.sum()), int(np.dot(j, j))
    mean = tr.value(Fraction(S, cnt))
    ss = Fraction(SS * cnt - S * S, cnt)                        # sum (j - mu)^2
    var = tr.scale ** 2 * F(ss) / (cnt - 1)
    if tr.delta == 0:
        mhat = _kernel_sum(float(tr.base) + float(tr.scale) * tr.j.astype(np.float64), lo, hi) / cnt
        eps = float(abs(mpf(mhat) - mean)) * SLACK + TINY
    else:
        mhat, eps = None, _mean_err(tr.xmax, mean, T)
    sc = abs(float(tr.scale))
    B2 = float(ss) * sc * sc
    B2in = float(ss) * (sc + 2 * tr.delta) ** 2                 # the device inputs' sum of squares, at most
    e = (B2in - B2) + cnt * eps * eps + gamma(-(-T // 32) + 35) * (B2in + cnt * eps * eps) + cnt * TINY
    e_var = (e / (cnt - 1) + U * (float(var) + e / (cnt - 1))) * SLACK
    return mean, eps + tr.delta, var, e_var, False, eps, mhat


class Ref:
    """the section 3.7 contract for one trace and max_lag, exactly, with the kernel's error bounds and every decision margin"""

    def __init__(self, tr, max_lag=0):
        T = self.T = tr.T
        whole, h1, h2 = tr.moments
        self.mean, self.e_mean, self.var, self.e_var, self.constant = whole[:5]
        self.halves = [h1[:4], h2[:4]]
        self.half_const = [h1[4], h2[4]]
        self.mhat = [whole[6], h1[6], h2[6]]                   # the device's means, where its inputs are exact
        self.margins = []                                       # (|value - boundary|, bound) of every decision taken
        self.ess, self.e_ess, self.lags, self.pairs, self.floor, self.cut = mpmath.nan, 0.0, 0, [], False, False
        self.defined = False
        if self.constant:
            return
        g = _geyer(tr)
        self.margins.append(g["g0 margin"])
        self.defined = g["defined"]
        if not self.defined:
            return
        L = min(T, max_lag) if max_lag > 0 else T
        m = min(len(g["pairs"]), L // 2)                        # pairs m need 2m + 1 < L
        self.margins += [p[2] for p in g["pairs"][:m]]
        self.cut = m == L // 2
        if not self.cut:
            self.margins.append(g["stop"])                      # the pair that turned non-positive
        self.pairs = [(p[0], p[1]) for p in g["pairs"][:m]]
        self.lags = 2 * m
        psum, e_sum, abs_sum = g["pairs"][m - 1][3:] if m else (Fraction(0), 0.0, 0.0)
        e_psum = e_sum + gamma(max(m, 1)) * abs_sum
        a = F(2 * psum - 1)
        e_a = 2 * e_psum + U * (abs(float(a)) + 2 * e_psum)
        f = 1 / mpmath.log10(T)
        e_f = gamma(6) * float(f)                               # device log10 within 1 ulp, then 1 / x
        self.margins.append((abs(float(a - f)), e_a + e_f))
        self.floor = f >= a
        tau, e_tau = (f, e_f) if self.floor else (a, e_a)
        self.ess = T / tau
        e = T * e_tau / (float(tau) * (float(tau) - e_tau))
        self.e_ess = (e + U * (float(self.ess) + e)) * SLACK


def _geyer(tr):
    """gamma_0 >= DBL_MIN, and Geyer's pairs without a max_lag cut up to the first non-positive one, with their bounds: per
    accepted pair (P, the previous pair, (|P|, its bound), then the running sum of the monotone pairs, the sum of their bounds
    and of their magnitudes)"""
    if tr.geyer is not None:
        return tr.geyer
    T, (whole, _, _) = tr.T, tr.moments
    sc, d = abs(float(tr.scale)), tr.delta
    eps_x = whole[5]                                            # the centring error of the device's mean
    # the kernel's g0 = fl(sum of staged squares / T), bounded in x units
    g0 = tr.scale ** 2 * tr.G2(0) / T ** 3
    sin = sc + 2 * d
    A0 = float(tr.G2(0)) / T ** 2 * sin * sin
    c = T * eps_x * eps_x                                       # sum_t (y_t - e)^2 = sum_t y_t^2 + T e^2
    e_g0 = float(g0) * ((sin / sc) ** 2 - 1) + (c + gamma(T + 2) * (A0 + c) + T * TINY) / T * (1 + gamma(2)) + U * float(g0) + TINY
    g = {"g0 margin": (abs(float(g0) - DBL_MIN), e_g0 * SLACK), "defined": g0 >= DBL_MIN, "pairs": [], "stop": None}
    if g["defined"]:
        eps = eps_x / (sc - 2 * d)                              # in units of j
        G0 = float(tr.G2(0)) / T ** 2
        psum, e_sum, abs_sum, prev, e_prev, m = Fraction(0), 0.0, 0.0, None, 0.0, 0
        while 2 * m + 1 < T:
            P = Fraction(tr.G2(2 * m) + tr.G2(2 * m + 1), tr.G2(0))
            e0, e1 = _e_rho(tr, 2 * m, eps, G0, sc - 2 * d), _e_rho(tr, 2 * m + 1, eps, G0, sc - 2 * d)
            eP = e0 + e1 + U * (abs(float(P)) + e0 + e1)
            if not P > 0:
                g["stop"] = (abs(float(P)), eP)
                break
            raw, before = P, prev
            if prev is not None and P > prev:
                P = prev
            e_prev = max(eP, e_prev)                            # |min(a', b') - min(a, b)| <= max(|a' - a|, |b' - b|)
            prev, psum, e_sum, abs_sum, m = P, psum + P, e_sum + e_prev, abs_sum + float(P) + e_prev, m + 1
            g["pairs"].append((raw, before, (abs(float(raw)), eP), psum, e_sum, abs_sum))
    tr.geyer = g
    return g


def _e_rho(tr, k, eps, G0, sc):
    """|rho^_k - rho_k|: the fma sum of the staged (x - m^) products in t order, the centring error eps (in units of j), the
    two divisions; sc is the device's level spacing at least"""
    while len(tr.E) <= k:
        i, T = len(tr.E), tr.T
        A = float(np.dot(tr.az[:T - i], tr.az[i:]))
        c = eps * tr.D(i) + (T - i) * eps * eps                 # sum (y_t - e)(y_{t+k} - e) - sum y_t y_{t+k}, at most
        tr.E.append((c + gamma(T + 2) * (A + c) + T * TINY / (sc * sc)) * SLACK)
    E0, Ek = tr.E[0], tr.E[k]
    assert E0 < G0 / 2, "gamma_0 is not resolved"
    rho = abs(tr.G2(k) / tr.G2(0))
    return ((Ek + rho * E0) / (G0 - E0) * (1 + gamma(3)) + gamma(3) * rho) * SLACK


def _far(ref, what):
    for value, bound in ref.margins:
        assert value > bound, ("a decision lies within its error bound of the boundary", what, value, bound)


def _kernel_order_sum(x):
    """pass 1's order: warp w sums t = w, w + 32, ... in t order, then one thread adds the 32 partials in warp order"""
    parts = [0.0] * 32
    for t, v in enumerate(x):
        parts[t % 32] += v
    s = 0.0
    for p in parts:
        s += p
    return s


# ----------------------------------------------------------------------------- crafted traces
T_LIST = (4, 5, 31, 32, 33, 63, 64, 65, 95, 96, 97, 128, 129, 2047, 2048)
GROUPS = ((2048, 2), (97, 3))          # extra chains of equal T with one shared layout: split-R-hat over each group
R = 2048                                # rows per chain in the store
SHAPES = (29, 30, 61, 62, 126)          # Q = 32, 33, 64, 65, 129
MAX_LAGS = (1, 2, 3, 31, 32, 33, 34, 63, 64, 65)


def _walk(rng, T, w, p):
    """reflecting walk on [0, w) that moves one step with probability p"""
    j, x = np.empty(T, np.int64), int(rng.integers(w))
    for t in range(T):
        if rng.random() < p:
            x = x + 1 if rng.random() < .5 else x - 1
            x = 1 if x < 0 else (w - 2 if x >= w else x)
        j[t] = x
    return j


def _two(rng, T, p_flip):
    """a 0/1 Markov trace that flips with probability p_flip, holding both values"""
    j = (np.cumsum(rng.random(T) < p_flip) + rng.integers(2)) % 2
    j[0], j[-1] = 0, 1
    return j


def _half_const(rng, T, first):
    n = T // 2
    j = rng.integers(0, 2, T)
    if first:
        j[:n], j[T - n], j[T - 1] = 0, 0, 1
    else:
        j[T - n:], j[0], j[n - 1] = 0, 1, 0
    return j


def _spike(T, t):
    j = np.zeros(T, np.int64)
    j[t] = 1
    return j


# integer site families: (name, positions used, j(rng, T)); the positions are disjoint, so one row is a permutation
SITE_FAMILIES = (
    ("white", 4, lambda rng, T: rng.integers(0, 4, T)),
    ("walk", 8, lambda rng, T: _walk(rng, T, 8, .08)),
    ("alternating", 2, lambda rng, T: np.arange(T) % 2),
    ("constant", 1, lambda rng, T: np.zeros(T, np.int64)),
    ("first half constant", 2, lambda rng, T: _half_const(rng, T, True)),
    ("second half constant", 2, lambda rng, T: _half_const(rng, T, False)),
    ("spike at 0", 2, lambda rng, T: _spike(T, 0)),
    ("spike at n - 1", 2, lambda rng, T: _spike(T, T // 2 - 1)),
    ("spike at T - 1", 2, lambda rng, T: _spike(T, T - 1)),
    ("spike at n", 2, lambda rng, T: _spike(T, T // 2)),        # the middle sample when T is odd: both halves constant
)


def _exp_levels(c0, c1):
    v = [mpmath.exp(mpf(c)) for c in (c0, c1)]
    delta = max(max(float(x) for x in v) * 2.0 ** -52, TINY)       # CUDA's double exp is within 1 ulp
    return float(c0), float(c1), v[0], v[1] - v[0], delta


def _ll(base, scale):
    """-loglik = base + scale * j on a grid where every value is an exact double"""
    def levels(j):
        x = np.float64(base) + np.float64(scale) * j
        for v in np.unique(j):
            assert Fraction(float(np.float64(base) + np.float64(scale) * v)) == Fraction(base) + Fraction(scale) * int(v)
        return base, scale, 0.0, -x
    return levels


# scalar families: (name, j(rng, T), levels); levels map j to (base, scale, delta, the stored doubles)
def _scalar_families():
    dy = 2.0 ** -30
    ll = (
        ("-loglik 1e5 walk", lambda rng, T: 37 * _walk(rng, T, 400, .9), _ll(1e5, dy)),
        ("-loglik 1e5 white", lambda rng, T: rng.integers(0, 1000, T), _ll(1e5, dy)),
        ("-loglik first half 0.1", lambda rng, T: _half_const(rng, T, True), _ll(0.1, 2.0 ** -4)),
        ("-loglik second half 0.1", lambda rng, T: _half_const(rng, T, False), _ll(0.1, 2.0 ** -4)),
        ("-loglik constant", lambda rng, T: np.zeros(T, np.int64), _ll(12345.678, 1.0)),
        ("-loglik 1e5 middle", lambda rng, T: 1000 * _spike(T, T // 2), _ll(1e5, dy)),
    )
    cd = []
    for name, c0, c1, fam in (("near 0 white", -1e-10, -3e-10, lambda rng, T: rng.integers(0, 2, T)),
                              ("near 0 sticky", -2e-10, -5e-10, lambda rng, T: _two(rng, T, .02)),
                              ("near -745", -745.0, -740.0, lambda rng, T: rng.integers(0, 2, T)),
                              ("alternating", -2.5, -0.7, lambda rng, T: np.arange(T) % 2),
                              ("constant", -1.3, -1.3, lambda rng, T: np.zeros(T, np.int64)),
                              ("first half constant", -0.2, -3.0, lambda rng, T: _half_const(rng, T, True))):
        lv = _exp_levels(c0, c1)
        cd.append((name, fam, lambda j, lv=lv: (lv[2], lv[3], lv[4], np.where(j == 0, lv[0], lv[1]))))
    return ll, tuple(cd)


LL_FAMILIES, CD_FAMILIES = _scalar_families()


def _resolved(make, T):
    """make() -> (j, Trace), drawn again until every decision of the trace, at every max_lag the tests use, lies farther from
    its boundary than the error bound (random traces only; a fixed one must pass at once)"""
    for _ in range(20):
        j, tr = make()
        if all(v > e for lag in (0,) + MAX_LAGS + (T - 1, T, T + 1) for v, e in Ref(tr, lag).margins):
            return j, tr
    raise AssertionError("no resolvable draw")


def _layout_for(rng, N):
    """family -> site; the last site (the tile that ends one quantity past a multiple of 32) and site 0 are always driven"""
    sites = [N - 1, 0] + list(rng.permutation(np.arange(1, N - 1))[:len(SITE_FAMILIES) - 2])
    return [int(s) for s in rng.permutation(sites)]


def _craft_chain(rng, N, T, layout, scalars):
    """R rows of pi (permutations) and cdl = (c, d, loglik), and the traces x_q of the chain's first T rows"""
    traces = {}
    pi = np.tile(np.arange(N, dtype=np.uint16), (R, 1))
    pos0 = 0
    for (name, width, fam), site in zip(SITE_FAMILIES, layout):
        j, tr = _resolved(lambda: (lambda j: (j, Trace(j, base=pos0)))(fam(rng, T)), T)
        assert 0 <= j.min() and j.max() < width
        pi[:T, site] = pos0 + j
        traces[3 + site] = (name, tr)
        pos0 += width
    # the other sites take the positions the driven sites leave in each row, in a random order
    driven = np.array(layout)
    free_sites = np.setdiff1d(np.arange(N), driven)
    taken = np.zeros((T, N), bool)
    taken[np.arange(T)[:, None], pi[:T, driven]] = True
    free = np.nonzero(~taken)[1].reshape(T, free_sites.size)
    while True:
        fill = np.take_along_axis(free, np.argsort(rng.random(free.shape), axis=1), axis=1)
        fillers = {3 + s: ("filler", Trace(fill[:, i])) for i, s in enumerate(free_sites)}
        if all(v > e for _, tr in fillers.values() for lag in (0,) + MAX_LAGS + (T - 1, T, T + 1) for v, e in Ref(tr, lag).margins):
            break
    pi[:T, free_sites] = fill
    traces.update(fillers)
    assert np.array_equal(np.sort(pi, axis=1), np.tile(np.arange(N), (R, 1)))
    cdl = np.zeros((R, 3))
    cdl[:, 2] = -1e5
    for q, fams, col in ((0, LL_FAMILIES, 2), (1, CD_FAMILIES, 0), (2, CD_FAMILIES, 1)):
        name, fam, levels = fams[scalars[q] % len(fams)]
        j, tr = _resolved(lambda: (lambda j: (j, Trace(j, *levels(j)[:3])))(fam(rng, T)), T)
        cdl[:T, col] = levels(j)[3]
        traces[q] = (name, tr)
    return pi, cdl, traces


@functools.lru_cache(maxsize=None)
def _crafted(N):
    """per chain: its own T, pi [R][N], cdl [R][3] and its traces; chains past the T sweep form the equal-T groups"""
    rng = np.random.default_rng(1000 + N)
    chains = []
    for idx, T in enumerate(T_LIST):
        chains.append((T,) + _craft_chain(rng, N, T, _layout_for(rng, N), (idx, idx + 2, idx + 4)))
    for T, k in GROUPS:                 # -loglik walk, exp(c) near 0 sticky, exp(d) alternating in every chain of a group
        layout = _layout_for(rng, N)
        for _ in range(k):
            chains.append((T,) + _craft_chain(rng, N, T, layout, (0, 1, 3)))
    return chains


@functools.lru_cache(maxsize=None)
def _ref(N, c, q, max_lag):
    T, _, _, traces = _crafted(N)[c]
    return Ref(traces[q][1], max_lag)


def _group_ids(N):
    ids, c = [], len(T_LIST)
    for T, k in GROUPS:
        ids.append((T, list(range(c, c + k))))
        c += k
    return ids


# ----------------------------------------------------------------------------- CPU: the reference itself
def test_exact_reference_equals_ref_stats_on_well_conditioned_traces():
    rng = np.random.default_rng(7)
    for T in (4, 5, 33, 97, 2048):
        for j in (rng.integers(0, 50, T), _walk(rng, T, 20, .3), _two(rng, T, .1), np.arange(T) % 3):
            x = j.astype(np.float64)
            for max_lag in (0, 1, 3, 33):
                mean, var, ess, lags, halves = ref_stats(x, max_lag)
                r = Ref(Trace(j), max_lag)
                assert r.lags == lags, (T, max_lag)
                got = [float(r.mean), float(r.var)] + [float(v) for h in r.halves for v in (h[0], h[2])]
                want = [mean, var, halves[0], halves[1], halves[2], halves[3]]
                assert np.allclose(got, want, rtol=1e-12, atol=0), (T, max_lag, got, want)
                assert abs(float(r.ess) / ess - 1) < 1e-9, (T, max_lag)


@pytest.mark.parametrize("phi", [0.0, 0.5, 0.9])
def test_exact_reference_on_ar1(phi):
    x = ar1(phi, 20_000, seed=int(phi * 10) + 1)
    j = np.round(x * 2 ** 16).astype(np.int64)                  # a dyadic grid: the doubles j / 2^16 are exact
    r = Ref(Trace(j, 0, 2.0 ** -16))
    mean, var, ess, lags, _ = ref_stats(j / 2.0 ** 16)
    assert r.lags == lags and abs(float(r.ess) / ess - 1) < 1e-9 and abs(float(r.var) / var - 1) < 1e-12
    tau = j.size / float(r.ess)
    assert abs(tau / ((1 + phi) / (1 - phi)) - 1) < 0.06, (phi, tau)


def test_error_bounds_are_tight_enough_to_see_a_one_pass_variance():
    """-loglik = 1e5 + j 2^-30: Sigma x^2 - T m^2 loses everything, and the bound on the two-pass form is far below that loss"""
    rng = np.random.default_rng(3)
    j = rng.integers(0, 1000, 2048)
    x = 1e5 + j * 2.0 ** -30
    r = Ref(Trace(j, 1e5, 2.0 ** -30))
    one_pass = (_kernel_order_sum(x * x) - x.size * (_kernel_order_sum(x) / x.size) ** 2) / (x.size - 1)
    assert abs(one_pass - float(r.var)) > 100 * r.e_var
    assert r.e_var < 1e-3 * float(r.var)


def test_crafted_traces_keep_every_decision_far_from_its_boundary():
    seen = dict(blocks=set(), floor=0, binds=0, undefined=0, inexact_half=0, exits=0)
    for N in SHAPES:
        chains = _crafted(N)
        for c, (T, _, cdl, traces) in enumerate(chains):
            Q = 3 + N
            for q in range(Q):
                for lag in (0,) + MAX_LAGS + (T - 1, T, T + 1):
                    r = _ref(N, c, q, lag)
                    _far(r, (N, c, q, lag))
                    if lag == 0 and r.defined:
                        seen["blocks"].add(r.lags // 32)
                        seen["floor"] += r.floor
                        seen["binds"] += any(p > prev and float(p - prev) > 1e-6 for p, prev in r.pairs if prev is not None)
                    seen["undefined"] += lag == 0 and not r.constant and not r.defined
            # warps of one tile leave at different lag blocks
            for q0 in range(0, Q, 32):
                stops = {_ref(N, c, q, 0).lags // 32 for q in range(q0, min(q0 + 32, Q)) if _ref(N, c, q, 0).defined}
                seen["exits"] += len(stops) > 1
            # a constant half of 0.1 whose kernel-order mean is not 0.1: dropping the constant-half rule shows
            name, tr = traces[0]
            if "0.1" in name:
                x = -cdl[:T, 2]
                h = x[:T // 2] if "first" in name else x[T - T // 2:T]
                seen["inexact_half"] += _kernel_order_sum(h) / h.size != h[0]
    assert max(seen["blocks"]) >= 3 and {0, 1, 2} <= seen["blocks"], seen
    assert seen["floor"] and seen["binds"] and seen["undefined"] and seen["inexact_half"] and seen["exits"], seen


# ----------------------------------------------------------------------------- GPU: crafted stores through a checkpoint
@pytest.fixture(scope="module")
def S():
    import seriation_b200 as S
    if not os.path.exists(S.LIB_PATH):
        S.build()
    S.lib()
    return S


def _crafted_run(S, tmp_path, N, store):
    """a real run of len(chains) chains and R rows, saved, its records overwritten with the crafted rows, loaded"""
    chains = _crafted(N)
    n = len(chains)
    X, hard = random_dataset(np.random.default_rng(N), N, 5, 2, .2)
    ds = S.Dataset.from_bits(X, hard)
    kw = dict(seed=11, store=store, max_samples=R)
    f = str(tmp_path / ("ck%d" % store))
    S.Run(ds, n, **kw).init().advance(R, True).save_checkpoint(f).close()
    for c, (T, pi, cdl, _) in enumerate(chains):
        def edit(rec, L, pi=pi, cdl=cdl, T=T):
            assert L["spi"] > 0 and (store == S.STORE_PI or L["sa"] > L["spi"])
            rec[L["spi"]:L["spi"] + pi.nbytes] = pi.tobytes()
            if store >= S.STORE_FULL:
                rec[L["cdl"]:L["cdl"] + cdl.nbytes] = cdl.tobytes()
            struct.pack_into("<i", rec, 156, T)
        patched = _patch_record(f, c, edit)                 # read in full before the file is truncated for writing
        with open(f, "wb") as out:
            out.write(patched)
    return S.Run(ds, n, **kw).load_checkpoint(f)


def _check(dg, col, N, c, qs, max_lag=0):
    T = _crafted(N)[c][0]
    assert dg["n_samples"][col] == T
    for q in qs:
        r, what = _ref(N, c, q, max_lag), (N, c, T, q, max_lag, _crafted(N)[c][3][q][0])
        got_h = dg["halves"][col, q]
        for got, want, e in ((dg["mean"][col, q], r.mean, r.e_mean), (dg["var"][col, q], r.var, r.e_var)) + tuple(
                (got_h[2 * i + k], r.halves[i][2 * k], r.halves[i][2 * k + 1]) for i in (0, 1) for k in (0, 1)):
            assert abs(mpf(float(got)) - want) <= e, what + (float(got), float(want), e)
        for i in (0, 1):
            if r.half_const[i]:
                assert got_h[2 * i + 1] == 0.0, what
        for got, want in zip((dg["mean"][col, q], got_h[0], got_h[2]), r.mhat):
            if want is not None:
                assert got == want, what + (got, want)
        if r.constant:
            assert dg["var"][col, q] == 0.0 and np.isnan(dg["ess"][col, q]) and dg["lags"][col, q] == 0, what
            continue
        assert dg["lags"][col, q] == (r.lags if r.defined else 0), what + (dg["lags"][col, q], r.lags)
        if not r.defined:
            assert np.isnan(dg["ess"][col, q]), what
        else:
            assert abs(mpf(float(dg["ess"][col, q])) - r.ess) <= r.e_ess, what + (dg["ess"][col, q], float(r.ess), r.e_ess)
            if r.cut:                                       # cut before a pair turned non-positive
                assert dg["lags"][col, q] == 2 * ((min(T, max_lag) if max_lag > 0 else T) // 2), what


def _rhat_interval(refs, n):
    """BDA3 over the exact halves' error boxes, with every host operation widened by its rounding: an interval"""
    iv = mpmath.iv
    iv.prec = 256
    rnd = lambda x: x * iv.mpf([1 - 2.0 ** -52, 1 + 2.0 ** -52])
    box = lambda v, e: iv.mpf([v - e, v + e])
    m = 2 * len(refs)
    W, mean = iv.mpf(0), iv.mpf(0)
    for r in refs:
        for h in r.halves:
            W = rnd(W + box(h[2], h[3]))
            mean = rnd(mean + box(h[0], h[1]))
    W, mean = rnd(W / m), rnd(mean / m)
    B = iv.mpf(0)
    for r in refs:
        for h in r.halves:
            d = rnd(box(h[0], h[1]) - mean)
            B = rnd(B + rnd(d * d))
    B = rnd(B / (m - 1))
    if W.a <= 0:
        return None
    nn = iv.mpf(n)
    return rnd(iv.sqrt(rnd(rnd(rnd(rnd(nn - 1) / nn) * W + B) / W)))


@pytest.mark.gpu
@pytest.mark.parametrize("N", SHAPES)
def test_crafted_traces_through_a_checkpoint(S, tmp_path, N):
    chains, Q = _crafted(N), 3 + N
    n = len(chains)
    run = _crafted_run(S, tmp_path, N, S.STORE_FULL)
    rng = np.random.default_rng(N)
    # about 40 ids: every chain, repeats, -1 and ids the run does not hold, in a random order
    chosen = np.array(list(rng.permutation(list(range(n)) + [0, n - 1, 3, 7, 3, -1, -1, n, n + 5, 999, -7] +
                                           list(rng.integers(0, n, 40 - n - 11)))), np.int32)
    both = run.diagnostics(chosen)
    for col, g in enumerate(chosen):
        if not 0 <= g < n:
            assert both["n_samples"][col] == 0 and np.all(np.isnan(both["mean"][col])) and np.all(np.isnan(both["halves"][col]))
            continue
        _check(both, col, N, int(g), range(Q))
    first = {int(g): col for col, g in enumerate(chosen) if 0 <= g < n}
    for col, g in enumerate(chosen):                          # a repeated id gives the same bits in every slab
        if 0 <= g < n:
            for key in ("mean", "var", "ess", "lags", "halves"):
                assert both[key][col].tobytes() == both[key][first[int(g)]].tobytes()
    # SCALARS only and SITES only: the same bits for the quantities each computes
    ids = np.arange(n, dtype=np.int32)
    full = run.diagnostics(ids)
    sc, si = run.diagnostics(ids, sites=False), run.diagnostics(ids, scalars=False)
    for key in ("mean", "var", "ess", "lags"):
        assert sc[key][:, :3].tobytes() == full[key][:, :3].tobytes() and np.all(np.isnan(sc[key][:, 3:])), key
        assert si[key][:, 3:].tobytes() == full[key][:, 3:].tobytes() and np.all(np.isnan(si[key][:, :3])), key
    # max_lag at the block edges, and at T - 1, T and T + 1 of each chain
    for lag in MAX_LAGS:
        dg = run.diagnostics(ids, max_lag=lag)
        for c in range(n):
            _check(dg, c, N, c, range(Q), lag)
    for c, (T, _, _, _) in enumerate(chains[:len(T_LIST)]):
        for lag in (T - 1, T, T + 1):
            _check(run.diagnostics([c], max_lag=lag), 0, N, c, range(Q), lag)
    # split-R-hat over chains of equal T against BDA3 on the exact halves; W = 0 gives NaN through the kernel
    nan_seen = 0
    for T, group in _group_ids(N):
        dg = run.diagnostics(np.array(group, np.int32))
        assert dg["rhat"] is not None
        for q in range(Q):
            refs = [_ref(N, c, q, 0) for c in group]
            box = _rhat_interval(refs, T // 2)
            if box is None:
                assert all(h[2] == 0 for r in refs for h in r.halves), (T, q)
                assert np.isnan(dg["rhat"][q]), (T, q)
                nan_seen += 1
            else:
                assert box.a <= dg["rhat"][q] <= box.b, (T, q, dg["rhat"][q], box)
    assert nan_seen
    # the same pi rows in a STORE_PI checkpoint: the sites' bits do not depend on the store or on `what`
    pi_run = _crafted_run(S, tmp_path, N, S.STORE_PI)
    pi_only = pi_run.diagnostics(ids, scalars=False)
    for key in ("mean", "var", "ess", "lags", "halves"):
        assert pi_only[key][:, 3:].tobytes() == full[key][:, 3:].tobytes(), key
    pi_run.close()
    run.close()


@pytest.mark.gpu
@pytest.mark.parametrize("big", [False, True], ids=["one-thread-per-taxon", "large-shape"])
def test_manycd_scalars_are_taxon_0(S, tmp_path, big):
    """on a manycd run q = 1, 2 are exp(c), exp(d) of taxon 0 (file order): the stored cdl row holds exactly c_all[:, 0]"""
    from conftest import load_hex_dataset
    ds = S.Dataset.from_bits(*load_hex_dataset("g10s10"))
    T = 40
    if big:
        os.environ["SER_FORCE_BIG"] = "256"
    try:
        run = S.Run(ds, 3, seed=8, manycd=True, store=S.STORE_FULL, max_samples=T).init().advance(T, True).sync()
    finally:
        os.environ.pop("SER_FORCE_BIG", None)
    assert (run.kernel_path() != 0) == big
    f = str(tmp_path / "m")
    run.save_checkpoint(f)
    data = open(f, "rb").read()
    size = struct.unpack_from("<Q", data, 88)[0]
    L = _layout(ds.N, ds.M, 1, S.STORE_FULL, T, 0)
    assert L["size"] == size
    first = 104 + (4 * 3 + 7) // 8 * 8 + 8
    dg = run.diagnostics([0, 1, 2], sites=False)
    for c in range(3):
        s = run.fetch_samples(c)
        cdl = np.frombuffer(data, np.float64, 3 * T, first + c * size + L["cdl"]).reshape(T, 3)
        assert cdl[:, 0].tobytes() == s["c_all"][:, 0].tobytes() == s["c"].tobytes(), c
        assert cdl[:, 1].tobytes() == s["d_all"][:, 0].tobytes() == s["d"].tobytes(), c
        assert np.ptp(s["c_all"][:, 0]) > 0 and np.ptp(s["d_all"][:, 0]) > 0
        for q, v in ((1, s["c_all"][:, 0]), (2, s["d_all"][:, 0])):
            want = mpmath.fsum(mpmath.exp(mpf(x)) for x in v) / T
            xmax = float(mpmath.exp(mpf(float(v.max()))))
            assert abs(mpf(float(dg["mean"][c, q])) - want) <= _mean_err(xmax * (1 + 2.0 ** -52), want, T) + xmax * 2.0 ** -52
    run.close()
