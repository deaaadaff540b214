"""ctypes binding of libseriation_b200.so (include/seriation_b200.h) plus a thin host-side mirror
of the reference's Python driver (script.py): ``run_all_chains``, ``choose_chains``,
``compute_pair_order_matrix`` keep their names and meaning, but run as one batched GPU launch.

The library is CUDA-only.  Loading fails loudly if it has not been built, and every compute call
raises ``SeriationError`` when no B200 is usable: there is no CPU fallback on this path.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SERIATION_B200_LIB") or os.path.join(HERE, "libseriation_b200.so")  # the override: instrumented builds

MODE_FREE, MODE_REPLAY = 0, 1
STORE_NONE, STORE_PI, STORE_FULL = 0, 1, 2
ACC_PO, ACC_SUMS, ACC_AB, ACC_ALIVE, ACC_POS, ACC_RANGE = 1, 2, 4, 8, 16, 32
DIAG_SCALARS, DIAG_SITES = 1, 2

_i32p, _dp, _u8p = C.POINTER(C.c_int32), C.POINTER(C.c_double), C.POINTER(C.c_uint8)
_i64p, _u64p = C.POINTER(C.c_int64), C.POINTER(C.c_uint64)


class SeriationError(RuntimeError):
    pass


class RunConfig(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_chains", C.c_int32), ("chain_offset", C.c_int32), ("sweeps_per_call", C.c_int32),
                ("mode", C.c_int32), ("seed", C.c_uint32), ("store", C.c_int32), ("max_samples", C.c_int32),
                ("device", C.c_int32), ("manycd", C.c_int32)]


# every symbol include/seriation_b200.h declares: (name, restype, argtypes)
_vp = C.c_void_p
SYMBOLS = [
    ("ser_last_error", C.c_char_p, []),
    ("ser_version", C.c_char_p, []),
    ("ser_dataset_from_bits", C.c_int, [C.c_int32, C.c_int32, _u8p, _u8p, C.POINTER(_vp)]),
    ("ser_dataset_read_txt", C.c_int, [C.c_char_p, C.POINTER(_vp)]),
    ("ser_dataset_read_stream", C.c_int, [_vp, C.POINTER(_vp)]),
    ("ser_dataset_dims", C.c_int, [_vp, _i32p, _i32p, _i32p]),
    ("ser_dataset_get", C.c_int, [_vp, _u8p, _u8p]),
    ("ser_dataset_free", None, [_vp]),
    ("ser_dataset_read_names", C.c_int, [_vp, C.c_char_p, C.c_char_p]),
    ("ser_dataset_taxon_name", C.c_char_p, [_vp, C.c_int32]),
    ("ser_dataset_site_name", C.c_char_p, [_vp, C.c_int32]),
    ("ser_dataset_site_age", C.c_int, [_vp, C.c_int32, _i32p, _dp, _i32p]),
    ("ser_dataset_synthetic", C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_uint64, C.POINTER(_vp)]),
    ("ser_run_create", C.c_int, [_vp, C.POINTER(RunConfig), C.POINTER(_vp)]),
    ("ser_run_create_chains", C.c_int, [_vp, C.POINTER(RunConfig), _i32p, C.c_int32, C.POINTER(_vp)]),
    ("ser_run_accumulate", C.c_int, [_vp, C.c_int32]),
    ("ser_run_destroy", None, [_vp]),
    ("ser_run_set_tapes", C.c_int, [_vp, _dp, _u64p]),
    ("ser_run_init", C.c_int, [_vp]),
    ("ser_run_advance", C.c_int, [_vp, C.c_int32, C.c_int32]),
    ("ser_run_advance_both", C.c_int, [_vp, C.c_int32, C.c_int32]),
    ("ser_run_sync", C.c_int, [_vp]),
    ("ser_run_elapsed_ms", C.c_int, [_vp, _dp, C.c_int32]),
    ("ser_run_kernel_launches", C.c_int, [_vp, _i64p]),
    ("ser_run_kernel_path", C.c_int, [_vp, _i32p]),
    ("ser_plan_warp_batches", C.c_int, [_i32p, C.c_int32, C.c_int32, _i32p, C.c_int32, _i32p]),
    ("ser_run_get_state", C.c_int, [_vp, C.c_int32] + [_i32p] * 9 + [_dp, _i64p]),
    ("ser_run_get_counters", C.c_int, [_vp, C.c_int32, _i64p]),
    ("ser_run_check", C.c_int, [_vp, _i32p]),
    ("ser_run_chain_stats", C.c_int, [_vp, _dp, _dp, _dp, _i32p]),
    ("ser_run_chain_stats_device", C.c_int, [_vp, _vp]),
    ("ser_run_fetch_samples", C.c_int, [_vp, C.c_int32, _i32p, _i32p, _i32p, _dp, _dp, _dp, _i32p]),
    ("ser_run_alive_counts", C.c_int, [_vp, _i32p, C.c_int32, _i32p, _i32p]),
    ("ser_run_get_flags", C.c_int, [_vp, C.c_int32, _i32p]),
    ("ser_run_get_cd", C.c_int, [_vp, C.c_int32, _dp, _dp]),
    ("ser_run_fetch_cd_samples", C.c_int, [_vp, C.c_int32, _dp, _dp, _i32p]),
    ("ser_select_chains", C.c_int, [_dp, C.c_int32, C.c_int32, _i32p, _i32p, _dp, _dp]),
    ("ser_select_chains_device", C.c_int, [_vp, C.c_int32, C.c_int32, _vp, _vp, C.c_int32, _vp]),
    ("ser_run_po_counts_device", C.c_int, [_vp, _vp, C.c_int32, _vp]),
    ("ser_run_po_counts", C.c_int, [_vp, _i32p, C.c_int32, _i32p]),
    ("ser_po_finalize", C.c_int, [_i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _dp]),
    ("ser_run_posterior_sums", C.c_int, [_vp, _i32p, C.c_int32, _i64p, _i32p, _i32p, _i32p, _i32p]),
    ("ser_run_diagnostics", C.c_int, [_vp, _i32p, C.c_int32, C.c_int32, C.c_int32, _dp, _dp, _i32p]),
    ("ser_split_rhat", C.c_int, [_dp, _i32p, C.c_int32, C.c_int32, _dp]),
    ("ser_run_marginals", C.c_int, [_vp, _i32p, C.c_int32, _i32p, _i32p, _i32p, _i32p]),
    ("ser_hist_quantiles", C.c_int, [_i32p, C.c_int32, C.c_int32, _dp, C.c_int32, _i32p]),
    ("ser_write_chain_files", C.c_int, [_vp, C.c_int32, C.c_char_p]),
    ("ser_write_labelled_files", C.c_int, [_vp, C.c_int32, _vp, C.c_char_p]),
    ("ser_microbench", C.c_int, [C.c_int32, _dp]),
    ("ser_microbench_ex", C.c_int, [C.c_int32, _dp]),
    ("ser_run_sweep_time", C.c_int, [_vp, _dp, _i32p, C.c_int32]),
    ("ser_run_site_age_corr", C.c_int, [_vp, _vp, _i32p, C.c_int32, _dp, _dp, _i32p]),
    ("ser_run_cross_chain_async", C.c_int, [_vp, _vp, C.c_int32]),
    ("ser_run_cross_chain_result", C.c_int, [_vp, _i32p, _i32p, _dp, _dp, _i32p]),
    ("ser_run_cross_chain_buffers", C.c_int, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    ("ser_comm_unique_id", C.c_int, [_u8p]),
    ("ser_comm_create", C.c_int, [_u8p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_vp)]),
    ("ser_comm_info", C.c_int, [_vp, _i32p, _i32p]),
    ("ser_comm_destroy", None, [_vp]),
    ("ser_multi_create", C.c_int, [_vp, C.POINTER(RunConfig), C.c_int32, _i32p, C.POINTER(_vp)]),
    ("ser_multi_destroy", None, [_vp]),
    ("ser_multi_init", C.c_int, [_vp]),
    ("ser_multi_advance", C.c_int, [_vp, C.c_int32, C.c_int32]),
    ("ser_multi_sync", C.c_int, [_vp]),
    ("ser_multi_elapsed_ms", C.c_int, [_vp, _dp, C.c_int32]),
    ("ser_multi_layout", C.c_int, [_vp, _i32p, _i32p, _i32p]),
    ("ser_multi_locate", C.c_int, [_vp, C.c_int32, C.POINTER(_vp), _i32p]),
    ("ser_multi_check", C.c_int, [_vp, _i32p]),
    ("ser_multi_chain_stats", C.c_int, [_vp, _dp, _dp, _dp, _i32p]),
    ("ser_multi_cross_chain", C.c_int, [_vp, C.c_int32, _i32p, _i32p, _dp, _dp, _i32p]),
    ("ser_run_save_checkpoint", C.c_int, [_vp, C.c_char_p]),
    ("ser_run_load_checkpoint", C.c_int, [_vp, C.c_char_p]),
    ("ser_multi_save_checkpoint", C.c_int, [_vp, C.c_char_p]),
    ("ser_multi_load_checkpoint", C.c_int, [_vp, C.c_char_p]),
    ("ser_checkpoint_info", C.c_int, [C.c_char_p, _i32p, _i32p, _i32p, _i64p, _i32p, C.POINTER(C.c_uint32), _i32p, _i32p]),
]
COMM_ID_BYTES = 128

_lib = None


def build() -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    subprocess.run(["sh", os.path.join(HERE, "build.sh")], check=True, stdout=subprocess.DEVNULL)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SeriationError(f"{LIB_PATH} is missing: run __graft_entry__.build() "
                                 "(there is no CPU fallback for the sweep)")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def _check(rc: int):
    if rc != 0:
        raise SeriationError(f"[{rc}] {lib().ser_last_error().decode()}")


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t)) if a is not None else None


def plan_warp_batches(ones_sorted, wcap: int) -> np.ndarray:
    """the warp batches of the large-shape kernel's Gibbs phase for sorted columns with these occurrence counts and slices of
    ``wcap`` items per warp (host only): rows of (first column, columns, lane shift, first item, last item + 1)"""
    ones = np.ascontiguousarray(ones_sorted, np.int32)
    n = C.c_int32()
    _check(lib().ser_plan_warp_batches(_p(ones, C.c_int32), ones.size, int(wcap), None, 0, C.byref(n)))
    raw = np.empty((n.value, 4), np.int32)
    _check(lib().ser_plan_warp_batches(_p(ones, C.c_int32), ones.size, int(wcap), _p(raw, C.c_int32), n.value, C.byref(n)))
    return np.stack([raw[:, 0], raw[:, 1] & 0xffff, raw[:, 1] >> 16, raw[:, 2], raw[:, 3]], axis=1)


class Dataset:
    """A sites x taxa 0/1 occurrence matrix with hard-site flags (the reference's .txt files)."""

    def __init__(self, handle):
        self._h = handle
        n, m, nh = C.c_int32(), C.c_int32(), C.c_int32()
        _check(lib().ser_dataset_dims(self._h, C.byref(n), C.byref(m), C.byref(nh)))
        self.N, self.M, self.nh = n.value, m.value, nh.value

    @classmethod
    def from_bits(cls, X, hard=None):
        X = np.ascontiguousarray(X, dtype=np.uint8)
        hard = np.zeros(X.shape[0], np.uint8) if hard is None else np.ascontiguousarray(hard, dtype=np.uint8)
        h = _vp()
        _check(lib().ser_dataset_from_bits(X.shape[0], X.shape[1], _p(X, C.c_uint8), _p(hard, C.c_uint8), C.byref(h)))
        return cls(h)

    @classmethod
    def read_txt(cls, path: str):
        h = _vp()
        _check(lib().ser_dataset_read_txt(path.encode(), C.byref(h)))
        return cls(h)

    @classmethod
    def synthetic(cls, N: int, M: int, n_hard: int = 16, seed: int = 0x5EB1A710):
        h = _vp()
        _check(lib().ser_dataset_synthetic(N, M, n_hard, seed, C.byref(h)))
        return cls(h)

    def read_names(self, genus_path=None, sites_path=None):
        _check(lib().ser_dataset_read_names(self._h, genus_path.encode() if genus_path else None,
                                            sites_path.encode() if sites_path else None))
        return self

    def taxon_name(self, m):
        s = lib().ser_dataset_taxon_name(self._h, m)
        return s.decode() if s else None

    def site_name(self, n):
        s = lib().ser_dataset_site_name(self._h, n)
        return s.decode() if s else None

    def site_age(self, n):
        mn, age, hard = C.c_int32(), C.c_double(), C.c_int32()
        _check(lib().ser_dataset_site_age(self._h, n, C.byref(mn), C.byref(age), C.byref(hard)))
        return mn.value, age.value, bool(hard.value)

    def arrays(self):
        X, hard = np.empty((self.N, self.M), np.uint8), np.empty(self.N, np.uint8)
        _check(lib().ser_dataset_get(self._h, _p(X, C.c_uint8), _p(hard, C.c_uint8)))
        return X, hard

    def __del__(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.ser_dataset_free(self._h)
            self._h = None


class Run:
    """A batch of independent chains on one GPU (replaces script.py's Pool of `mcmc` processes).  ``chain_ids``: the global
    ids of the local chains (a subset run, ser_run_create_chains; ``n_chains`` is then ignored)."""

    def __init__(self, ds: Dataset, n_chains: int, *, mode=MODE_FREE, seed=0, chain_offset=0, sweeps_per_call=10,
                 store=STORE_NONE, max_samples=0, device=0, manycd=False, chain_ids=None):
        self.ds = ds
        ids = None if chain_ids is None else np.ascontiguousarray(chain_ids, dtype=np.int32)
        if ids is not None:
            n_chains = ids.size
        self.N, self.M, self.n_chains = ds.N, ds.M, n_chains
        self.manycd = bool(manycd)
        self.cfg = RunConfig(C.sizeof(RunConfig), n_chains, chain_offset, sweeps_per_call, mode, seed, store, max_samples, device,
                             int(self.manycd))
        h = _vp()
        if ids is None:
            _check(lib().ser_run_create(ds._h, C.byref(self.cfg), C.byref(h)))
        else:
            _check(lib().ser_run_create_chains(ds._h, C.byref(self.cfg), _p(ids, C.c_int32), ids.size, C.byref(h)))
        self._h = h

    def accumulate(self, po=True, sums=True, ab=False, alive=False, positions=False, ranges=False):
        """from now on the sample store is a window of max_samples rows and the summaries sum over every sample taken
        afterwards (ser_run_accumulate); call before the first sampling call.  ``positions`` / ``ranges`` accumulate the
        histograms of marginals()"""
        what = (ACC_PO if po else 0) | (ACC_SUMS if sums else 0) | (ACC_AB if ab else 0) | (ACC_ALIVE if alive else 0)
        what |= (ACC_POS if positions else 0) | (ACC_RANGE if ranges else 0)
        _check(lib().ser_run_accumulate(self._h, what))
        return self

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.ser_run_destroy(self._h)
            self._h = None

    __del__ = close

    def set_tapes(self, tapes):
        """tapes: list of 1-D float64 arrays, one per local chain (replay mode)."""
        offs = np.zeros(len(tapes) + 1, np.uint64)
        offs[1:] = np.cumsum([t.size for t in tapes])
        flat = np.ascontiguousarray(np.concatenate(tapes), dtype=np.float64)
        _check(lib().ser_run_set_tapes(self._h, _p(flat, C.c_double), _p(offs, C.c_uint64)))
        return self

    def init(self):
        _check(lib().ser_run_init(self._h))
        return self

    def save_checkpoint(self, path):
        """every chain's state (and stored samples, accumulators) to ``path``, written atomically (ser_run_save_checkpoint)"""
        _check(lib().ser_run_save_checkpoint(self._h, os.fsencode(path)))
        return self

    def load_checkpoint(self, path):
        """in place of init(): continue the chains saved in ``path`` bit for bit (set_tapes / accumulate come first)"""
        _check(lib().ser_run_load_checkpoint(self._h, os.fsencode(path)))
        return self

    def advance(self, n_calls: int, sampling: bool):
        _check(lib().ser_run_advance(self._h, n_calls, int(sampling)))
        return self

    def advance_both(self, burn_calls: int, sample_calls: int):
        """burn-in calls, then sampling calls, in one launch (main's two loops, mcmc.c:140-143 + :180-185)"""
        _check(lib().ser_run_advance_both(self._h, burn_calls, sample_calls))
        return self

    def sync(self):
        _check(lib().ser_run_sync(self._h))
        return self

    def elapsed_ms(self, reset=False) -> float:
        ms = C.c_double()
        _check(lib().ser_run_elapsed_ms(self._h, C.byref(ms), int(reset)))
        return ms.value

    def sweep_time(self, reset=False):
        """(ms, launches): CUDA-event time of the sweep launches alone since the last reset"""
        ms, n = C.c_double(), C.c_int32()
        _check(lib().ser_run_sweep_time(self._h, C.byref(ms), C.byref(n), int(reset)))
        return ms.value, n.value

    def kernel_launches(self) -> int:
        n = C.c_int64()
        _check(lib().ser_run_kernel_launches(self._h, C.byref(n)))
        return n.value

    def kernel_path(self) -> int:
        """0 = one thread per taxon, 1 = large-shape kernel (CTA-wide column groups), 2 = large-shape kernel (warp batches)"""
        n = C.c_int32()
        _check(lib().ser_run_kernel_path(self._h, C.byref(n)))
        return n.value

    def state(self, chain: int) -> dict:
        N, M = self.N, self.M
        a, b, t0, f0, t1, f1 = (np.empty(M, np.int32) for _ in range(6))
        pi, rpi = np.empty(N, np.int32), np.empty(N, np.int32)
        tot, cdl, slots = np.empty(4, np.int32), np.empty(3), C.c_int64()
        _check(lib().ser_run_get_state(self._h, chain, *(_p(v, C.c_int32) for v in (a, b, pi, rpi, t0, f0, t1, f1, tot)),
                                       _p(cdl, C.c_double), C.byref(slots)))
        return dict(a=a, b=b, pi=pi, rpi=rpi, t0=t0, f0=f0, t1=t1, f1=f1, tot=tot, c=cdl[0], d=cdl[1],
                    loglik=cdl[2], slots=slots.value)

    def cd(self, chain: int):
        """per-taxon (c, d) of a manycd run, file order"""
        c, d = np.empty(self.M), np.empty(self.M)
        _check(lib().ser_run_get_cd(self._h, chain, _p(c, C.c_double), _p(d, C.c_double)))
        return c, d

    def counters(self, chain: int) -> np.ndarray:
        out = np.empty(8, np.int64)
        _check(lib().ser_run_get_counters(self._h, chain, _p(out, C.c_int64)))
        return out

    def check(self) -> int:
        bad = C.c_int32()
        rc = lib().ser_run_check(self._h, C.byref(bad))
        if rc not in (0, -7):
            _check(rc)
        return bad.value

    def flags(self, chain: int) -> int:
        f = C.c_int32()
        _check(lib().ser_run_get_flags(self._h, chain, C.byref(f)))
        return f.value

    def chain_stats(self):
        e, c, d = (np.empty(self.n_chains) for _ in range(3))
        n = C.c_int32()
        _check(lib().ser_run_chain_stats(self._h, _p(e, C.c_double), _p(c, C.c_double), _p(d, C.c_double), C.byref(n)))
        return dict(e_negloglik=e, e_c=c, e_d=d, n_samples=n.value)

    def chain_stats_device(self, device_ptr: int):
        _check(lib().ser_run_chain_stats_device(self._h, device_ptr))

    def fetch_samples(self, chain: int, full=True) -> dict:
        n = C.c_int32()
        _check(lib().ser_run_fetch_samples(self._h, chain, None, None, None, None, None, None, C.byref(n)))
        S, N, M = n.value, self.N, self.M
        pi = np.empty((S, N), np.int32)
        if not full:
            _check(lib().ser_run_fetch_samples(self._h, chain, None, None, _p(pi, C.c_int32), None, None, None, C.byref(n)))
            return dict(pi=pi)
        a, b = np.empty((S, M), np.int32), np.empty((S, M), np.int32)
        c, d, ll = np.empty(S), np.empty(S), np.empty(S)
        _check(lib().ser_run_fetch_samples(self._h, chain, _p(a, C.c_int32), _p(b, C.c_int32), _p(pi, C.c_int32),
                                           _p(c, C.c_double), _p(d, C.c_double), _p(ll, C.c_double), C.byref(n)))
        out = dict(a=a, b=b, pi=pi, c=c, d=d, loglik=ll)
        if self.manycd:
            c_all, d_all = np.empty((S, M)), np.empty((S, M))
            _check(lib().ser_run_fetch_cd_samples(self._h, chain, _p(c_all, C.c_double), _p(d_all, C.c_double), C.byref(n)))
            out.update(c_all=c_all, d_all=d_all)
        return out

    def po_counts(self, chosen) -> np.ndarray:
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        out = np.zeros((len(chosen), self.N, self.N), np.int32)
        _check(lib().ser_run_po_counts(self._h, _p(chosen, C.c_int32), len(chosen), _p(out, C.c_int32)))
        return out

    def posterior_sums(self, chosen, with_ab: bool = False) -> dict:
        """per chosen chain: sum_t sum_i i*pi_t(i), sum_t pi_t, (sum_t a_t, sum_t b_t) over the stored samples"""
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        k = len(chosen)
        corr, pi_sum = np.zeros(k, np.int64), np.zeros((k, self.N), np.int32)
        a_sum = np.zeros((k, self.M), np.int32) if with_ab else None
        b_sum = np.zeros((k, self.M), np.int32) if with_ab else None
        n = C.c_int32()
        _check(lib().ser_run_posterior_sums(self._h, _p(chosen, C.c_int32), k, _p(corr, C.c_int64), _p(pi_sum, C.c_int32),
                                            _p(a_sum, C.c_int32), _p(b_sum, C.c_int32), C.byref(n)))
        return dict(corr_num=corr, pi_sum=pi_sum, a_sum=a_sum, b_sum=b_sum, n_samples=n.value)

    def alive_counts(self, chosen) -> tuple:
        """int32 [k][N][M]: #{t: a_t(m) <= j <= b_t(m)} per chosen chain, and the number of samples T"""
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        out, n = np.zeros((len(chosen), self.N, self.M), np.int32), C.c_int32()
        _check(lib().ser_run_alive_counts(self._h, _p(chosen, C.c_int32), len(chosen), _p(out, C.c_int32), C.byref(n)))
        return out, n.value

    def diagnostics(self, chosen, scalars: bool = True, sites: bool = True, max_lag: int = 0) -> dict:
        """convergence diagnostics of the chosen chains (global ids) over their stored samples (ser_run_diagnostics): per chain and
        quantity (Q = 3 + N: -loglik, exp(c), exp(d), then pi of every site) ``mean``, ``var``, ``ess``, ``lags`` [k][Q], ``halves``
        [k][Q][4] (mean1, var1, mean2, var2), ``n_samples`` [k] and the split ``rhat`` [Q] over the chains this run holds (None when
        their sample counts differ).  Slabs the run does not fill stay NaN (n_samples 0)."""
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        k, Q = len(chosen), 3 + self.N
        stats, halves = np.full((k, Q, 4), np.nan), np.full((k, Q, 4), np.nan)
        n = np.zeros(k, np.int32)
        what = (DIAG_SCALARS if scalars else 0) | (DIAG_SITES if sites else 0)
        _check(lib().ser_run_diagnostics(self._h, _p(chosen, C.c_int32), k, what, int(max_lag), _p(stats, C.c_double),
                                         _p(halves, C.c_double), _p(n, C.c_int32)))
        held = n > 0
        rhat = split_rhat(halves[held], n[held]) if held.any() and np.all(n[held] == n[held][0]) else None
        return dict(mean=stats[..., 0], var=stats[..., 1], ess=stats[..., 2], lags=stats[..., 3], halves=halves, n_samples=n, rhat=rhat)

    def marginals(self, chosen, ranges: bool = False, positions: bool = True) -> dict:
        """histograms of the chosen chains (global ids) over their samples (ser_run_marginals): ``pos`` [k][N][N] = #{t: pi_t(i) = p},
        and with ``ranges`` ``a`` / ``b`` [k][M][N+1] = #{t: a_t(m) = j}; ``n_samples`` [k] = T.  Slabs the run does not fill stay 0
        (n_samples 0)."""
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        k, N, M = len(chosen), self.N, self.M
        pos = np.zeros((k, N, N), np.int32) if positions else None
        a = np.zeros((k, M, N + 1), np.int32) if ranges else None
        b = np.zeros((k, M, N + 1), np.int32) if ranges else None
        n = np.zeros(k, np.int32)
        _check(lib().ser_run_marginals(self._h, _p(chosen, C.c_int32), k, _p(pos, C.c_int32), _p(a, C.c_int32), _p(b, C.c_int32),
                                       _p(n, C.c_int32)))
        return dict(pos=pos, a=a, b=b, n_samples=n)

    def po_counts_device(self, chosen_ptr: int, k: int, counts_ptr: int):
        _check(lib().ser_run_po_counts_device(self._h, chosen_ptr, k, counts_ptr))

    def cross_chain_async(self, k: int, comm=None):
        """E[-logL] -> (all-gather) -> choose_chains(k) -> pair-order counts -> (all-reduce), enqueued on the
        run's stream without any host synchronisation; ``comm``: a Comm when the chains are sharded over ranks"""
        _check(lib().ser_run_cross_chain_async(self._h, comm._h if comm is not None else None, k))
        self._cc_k = k
        return self

    def cross_chain_result(self, with_counts: bool = True):
        k = self._cc_k
        chosen, n = np.empty(k, np.int32), C.c_int32()
        mn, sd = C.c_double(), C.c_double()
        counts = np.empty((k, self.N, self.N), np.int32) if with_counts else None
        _check(lib().ser_run_cross_chain_result(self._h, _p(chosen, C.c_int32), C.byref(n), C.byref(mn), C.byref(sd),
                                                _p(counts, C.c_int32)))
        return dict(chosen=chosen[:n.value].copy(), min=mn.value, sigma=sd.value, counts=counts)

    def cross_chain(self, k: int, comm=None, with_counts: bool = True):
        return self.cross_chain_async(k, comm).cross_chain_result(with_counts)

    def site_age_corr(self, chosen):
        """CORR_MN: mean over the stored samples of pearsonr(pi_t, x), x = -age_ma and x = MN unit of the
        .sites file (the dataset needs read_names); returns (corr_age, corr_mn)"""
        chosen = np.ascontiguousarray(chosen, dtype=np.int32)
        ca, cm, n = C.c_double(), C.c_double(), C.c_int32()
        _check(lib().ser_run_site_age_corr(self._h, self.ds._h, _p(chosen, C.c_int32), len(chosen), C.byref(ca), C.byref(cm), C.byref(n)))
        return ca.value, cm.value

    def write_chain_files(self, chain: int, directory: str):
        _check(lib().ser_write_chain_files(self._h, chain, directory.encode()))

    def write_labelled_files(self, chain: int, directory: str):
        _check(lib().ser_write_labelled_files(self._h, chain, self.ds._h, directory.encode()))


class _BorrowedRun(Run):
    """a ser_run owned by a Multi (never destroyed from Python)"""

    def __init__(self, handle, ds, n_chains, manycd):
        self._h, self.ds, self.N, self.M, self.n_chains, self.manycd = handle, ds, ds.N, ds.M, n_chains, manycd

    def close(self):
        self._h = None

    __del__ = close


class Comm:
    """NCCL communicator of one rank (one process per GPU).  ``Comm.unique_id()`` on rank 0, broadcast the 128
    bytes with whatever launched the ranks (torch.distributed, MPI, a file), then ``Comm(id, n_ranks, rank, device)``."""

    @staticmethod
    def unique_id() -> bytes:
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        _check(lib().ser_comm_unique_id(buf))
        return bytes(buf)

    def __init__(self, uid: bytes, n_ranks: int, rank: int, device: int = 0):
        assert len(uid) == COMM_ID_BYTES
        buf = (C.c_uint8 * COMM_ID_BYTES).from_buffer_copy(uid)
        h = _vp()
        _check(lib().ser_comm_create(buf, n_ranks, rank, device, C.byref(h)))
        self._h, self.n_ranks, self.rank = h, n_ranks, rank

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.ser_comm_destroy(self._h)
            self._h = None

    __del__ = close


class Multi:
    """All chains of one call sharded over the GPUs of one box by ONE process (run_all_chains' Pool, script.py:48-67)."""

    def __init__(self, ds: Dataset, n_chains: int, n_gpus: int, *, seed=0, chain_offset=0, sweeps_per_call=10, store=STORE_PI,
                 max_samples=0, manycd=False, devices=None):
        self.ds, self.N, self.M, self.n_chains, self.n_gpus, self.first = ds, ds.N, ds.M, n_chains, n_gpus, chain_offset
        self.manycd = bool(manycd)
        cfg = RunConfig(C.sizeof(RunConfig), n_chains, chain_offset, sweeps_per_call, MODE_FREE, seed, store, max_samples, 0, int(self.manycd))
        dev = np.ascontiguousarray(devices, dtype=np.int32) if devices is not None else None
        h = _vp()
        _check(lib().ser_multi_create(ds._h, C.byref(cfg), n_gpus, _p(dev, C.c_int32), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None) and _lib is not None:
            _lib.ser_multi_destroy(self._h)
            self._h = None

    __del__ = close

    def init(self):
        _check(lib().ser_multi_init(self._h))
        return self

    def advance(self, burn_calls: int, sample_calls: int):
        _check(lib().ser_multi_advance(self._h, burn_calls, sample_calls))
        return self

    def save_checkpoint(self, path):
        """every device's chains to one file, in global order (ser_multi_save_checkpoint)"""
        _check(lib().ser_multi_save_checkpoint(self._h, os.fsencode(path)))
        return self

    def load_checkpoint(self, path):
        """in place of init(): each device reads its own chains' records from ``path``"""
        _check(lib().ser_multi_load_checkpoint(self._h, os.fsencode(path)))
        return self

    def sync(self):
        _check(lib().ser_multi_sync(self._h))
        return self

    def elapsed_ms(self, reset=False) -> float:
        ms = C.c_double()
        _check(lib().ser_multi_elapsed_ms(self._h, C.byref(ms), int(reset)))
        return ms.value

    def layout(self) -> dict:
        n, per, peer = C.c_int32(), np.zeros(8, np.int32), C.c_int32()
        _check(lib().ser_multi_layout(self._h, C.byref(n), _p(per, C.c_int32), C.byref(peer)))
        return dict(n_gpus=n.value, chains_per_gpu=per[:n.value].tolist(), peer_stores=bool(peer.value))

    def locate(self, global_chain: int):
        """(Run view, local chain index) of a global chain id"""
        h, loc = _vp(), C.c_int32()
        _check(lib().ser_multi_locate(self._h, global_chain, C.byref(h), C.byref(loc)))
        return _BorrowedRun(h, self.ds, self.n_chains, self.manycd), loc.value

    def check(self) -> int:
        bad = C.c_int32()
        rc = lib().ser_multi_check(self._h, C.byref(bad))
        if rc not in (0, -7):
            _check(rc)
        return bad.value

    def chain_stats(self):
        e, c, d = (np.empty(self.n_chains) for _ in range(3))
        n = C.c_int32()
        _check(lib().ser_multi_chain_stats(self._h, _p(e, C.c_double), _p(c, C.c_double), _p(d, C.c_double), C.byref(n)))
        return dict(e_negloglik=e, e_c=c, e_d=d, n_samples=n.value)

    def cross_chain(self, k: int, with_counts: bool = True):
        chosen, n = np.empty(k, np.int32), C.c_int32()
        mn, sd = C.c_double(), C.c_double()
        counts = np.empty((k, self.N, self.N), np.int32) if with_counts else None
        _check(lib().ser_multi_cross_chain(self._h, k, _p(chosen, C.c_int32), C.byref(n), C.byref(mn), C.byref(sd), _p(counts, C.c_int32)))
        return dict(chosen=chosen[:n.value].copy(), min=mn.value, sigma=sd.value, counts=counts)


def select_chains(e_negloglik, k: int):
    """choose_chains (script.py:70-99) on the host. Returns (sorted ids, min, sigma)."""
    e = np.ascontiguousarray(e_negloglik, dtype=np.float64)
    chosen, n = np.empty(max(k, 1), np.int32), C.c_int32()
    mn, sd = C.c_double(), C.c_double()
    _check(lib().ser_select_chains(_p(e, C.c_double), e.size, k, _p(chosen, C.c_int32), C.byref(n), C.byref(mn), C.byref(sd)))
    return chosen[:n.value].copy(), mn.value, sd.value


def checkpoint_info(path) -> dict:
    """the header of a checkpoint file (host only, no CUDA call): what a resume needs to plan the remaining calls"""
    n, m, nc, ns, mode, many = (C.c_int32() for _ in range(6))
    calls, seed = C.c_int64(), C.c_uint32()
    _check(lib().ser_checkpoint_info(os.fsencode(path), C.byref(n), C.byref(m), C.byref(nc), C.byref(calls), C.byref(ns), C.byref(seed),
                                     C.byref(mode), C.byref(many)))
    return dict(N=n.value, M=m.value, n_chains=nc.value, calls_done=calls.value, n_samples=ns.value, seed=seed.value, mode=mode.value,
                manycd=bool(many.value))


def split_rhat(halves, n_samples) -> np.ndarray:
    """split-R-hat per quantity from the [k][Q][4] halves of k chains with equal sample counts (ser_split_rhat, host only)"""
    halves = np.ascontiguousarray(halves, dtype=np.float64)
    n = np.ascontiguousarray(n_samples, dtype=np.int32)
    k, Q = halves.shape[0], halves.shape[1]
    out = np.empty(Q)
    _check(lib().ser_split_rhat(_p(halves, C.c_double), _p(n, C.c_int32), k, Q, _p(out, C.c_double)))
    return out


def hist_quantiles(hist, probs) -> np.ndarray:
    """per row of ``hist`` [..., bins] the smallest bin whose cumulative count reaches p * total for each p in ``probs``
    (numpy's "inverted_cdf"; -1 for an empty row), [..., len(probs)] (ser_hist_quantiles, host only)"""
    h = np.ascontiguousarray(hist, dtype=np.int32)
    p = np.ascontiguousarray(np.atleast_1d(probs), dtype=np.float64)
    bins = h.shape[-1]
    rows = h.size // bins if bins else 0
    out = np.empty(h.shape[:-1] + (p.size,), np.int32)
    _check(lib().ser_hist_quantiles(_p(h, C.c_int32), rows, bins, _p(p, C.c_double), p.size, _p(out, C.c_int32)))
    return out


def select_chains_device(e_ptr: int, n: int, k: int, chosen_ptr: int, info_ptr: int, device=0, stream=None):
    _check(lib().ser_select_chains_device(e_ptr, n, k, chosen_ptr, info_ptr, device, stream))


def po_finalize(counts: np.ndarray, chains_selected: int, faithful=True) -> np.ndarray:
    counts = np.ascontiguousarray(counts, dtype=np.int32)
    k, N, _ = counts.shape
    po = np.empty((N, N))
    _check(lib().ser_po_finalize(_p(counts, C.c_int32), k, N, chains_selected, int(faithful), _p(po, C.c_double)))
    return po


def microbench(device=0) -> dict:
    out = np.empty(6)
    _check(lib().ser_microbench_ex(device, _p(out, C.c_double)))
    return dict(fp64_tflops=out[0], lds_gbs=out[1], popc_gops=out[2], fp64_kernel_ms=out[3], lds_kernel_ms=out[4], popc_kernel_ms=out[5])


# ------------------------------------------------------------------------------------------------
# host-side mirror of script.py
class ChainBatch:
    """What ``run_all_chains(dataset)`` leaves behind in the reference -- 100 ``Chains/chain_XX/``
    directories -- kept on the GPU instead: E[-logL] per chain and the pi history."""

    def __init__(self, run: Run, burn_calls: int, sample_calls: int, *, seed: int = 0, sweeps_per_call: int = 10,
                 manycd: bool = False):
        self.run, self.burn_calls, self.sample_calls = run, burn_calls, sample_calls
        self.seed, self.sweeps_per_call, self.manycd = seed, sweeps_per_call, manycd   # what replay_chosen rebuilds the chains from
        self._stats = None

    def stats(self):
        if self._stats is None:
            self._stats = self.run.chain_stats()
        return self._stats


def run_all_chains(dataset, n_chains: int = 100, burn_calls: int = 1000, sample_calls: int = 1000, *, seed: int = 0,
                   device: int = 0, store: int = STORE_PI, chains_dir: str | None = None) -> ChainBatch:
    """script.py:48-67.  ``dataset`` is a path to a reference .txt file or a Dataset.  One launch
    simulates all chains (the reference: Pool(8) over 100 ``./mcmc <i> < dataset`` processes).
    With ``chains_dir`` the reference's per-chain files are written for the first 100 chains."""
    ds = dataset if isinstance(dataset, Dataset) else Dataset.read_txt(str(dataset))
    if chains_dir is not None:
        store = STORE_FULL
    run = Run(ds, n_chains, mode=MODE_FREE, seed=seed, store=store, max_samples=sample_calls, device=device)
    run.init().advance(burn_calls, False).advance(sample_calls, True).sync()
    batch = ChainBatch(run, burn_calls, sample_calls, seed=seed, sweeps_per_call=run.cfg.sweeps_per_call, manycd=run.manycd)
    if chains_dir is not None:
        for i in range(min(n_chains, 100)):
            d = os.path.join(chains_dir, "chain_%02d" % i)
            os.makedirs(d, exist_ok=True)
            run.write_chain_files(i, d)
    return batch


def choose_chains(batch: ChainBatch, chains_selected: int):
    """script.py:70-99 over the batch's E[-logL]."""
    chosen, _, _ = select_chains(batch.stats()["e_negloglik"], chains_selected)
    return [int(c) for c in chosen]


def replay_chosen(batch: ChainBatch, chains, *, window: int = 64, with_ab: bool = False, marginals: bool = False,
                  device=None) -> ChainBatch:
    """The second phase of select-then-replay: re-simulate the chosen chains of a batch (typically one run with
    ``store=STORE_NONE``, which holds no sample history) alone, bit for bit, while their summaries accumulate through a
    ``window``-row sample store.  The returned batch's ``run`` is that subset run and its ``stats()`` are the first
    run's, so compute_pair_order_matrix, compute_exp_* and the probability maps work on it unchanged.  ``with_ab``
    also accumulates the a/b sums and alive counts (compute_exp_a and the maps need them).  ``window=0`` keeps every
    sample instead (``STORE_FULL``, no accumulators): the summaries take the one-shot path and ``diagnostics`` works on
    the result.  ``marginals`` also accumulates the position and a/b histograms of marginals() (the window then keeps a and b).
    Raises SeriationError when a replayed chain's E[-logL] differs from its first run in any bit."""
    ids = np.ascontiguousarray(chains, dtype=np.int32)
    keep_all = window == 0
    run = Run(batch.run.ds, ids.size, seed=batch.seed, sweeps_per_call=batch.sweeps_per_call, manycd=batch.manycd,
              store=STORE_FULL if (with_ab or keep_all or marginals) else STORE_PI, max_samples=batch.sample_calls if keep_all else window,
              device=batch.run.cfg.device if device is None else device, chain_ids=ids)
    run.init()
    if not keep_all:
        run.accumulate(po=True, sums=True, ab=with_ab, alive=with_ab, positions=marginals, ranges=marginals)
    run.advance(batch.burn_calls, False).advance(batch.sample_calls, True).sync()
    want, got = batch.stats()["e_negloglik"][ids], run.chain_stats()["e_negloglik"]
    if want.tobytes() != got.tobytes():
        raise SeriationError(f"replay_chosen: the replayed chains {ids.tolist()} do not reproduce their first run "
                             f"(E[-logL] {got.tolist()} vs {want.tolist()})")
    out = ChainBatch(run, batch.burn_calls, batch.sample_calls, seed=batch.seed, sweeps_per_call=batch.sweeps_per_call,
                     manycd=batch.manycd)
    out._stats = batch.stats()
    return out


def compute_pair_order_matrix(batch: ChainBatch, chains, chains_selected: int, sites: int | None = None, faithful=True):
    """script.py:155-189 for the chosen chains; counts on the GPU, the reference's division quirks on
    the host.  ``sites`` is accepted for signature compatibility."""
    counts = batch.run.po_counts(np.asarray(chains, dtype=np.int32))
    return po_finalize(counts, chains_selected, faithful)


def diagnostics(batch: ChainBatch, chains, max_lag: int = 0) -> dict:
    """Run.diagnostics over the chosen chains of a batch: every site's pi, and -loglik, exp(c), exp(d) when the batch keeps the
    full sample store (their rows stay NaN otherwise).  A batch from replay_chosen(..., window=0) keeps it."""
    run = batch.run
    return run.diagnostics(np.asarray(chains, dtype=np.int32), scalars=run.cfg.store >= STORE_FULL, max_lag=max_lag)


def _marginal_summary(hist, probs):
    """mean, quantiles [rows][len(probs)], mode and P(mode) of every row of pooled counts [rows][bins]"""
    total = hist.sum(axis=1, dtype=np.int64)
    mean = (hist.astype(np.int64) @ np.arange(hist.shape[1], dtype=np.int64)) / total
    mode = hist.argmax(axis=1)
    return dict(mean=mean, quantiles=hist_quantiles(hist, probs), mode=mode, p_mode=hist[np.arange(len(hist)), mode] / total)


def marginals(batch: ChainBatch, chains, probs=(0.025, 0.5, 0.975)) -> dict:
    """Posterior marginals pooled over the chosen chains by summing their counts: per site (file order) the position's ``mean``,
    ``quantiles`` [N][len(probs)], ``mode`` and ``p_mode``, in ``sites``; per taxon the same for a and for b, in ``a`` and ``b``
    (None unless the batch keeps a and b: the full sample store, or replay_chosen(..., marginals=True)).  ``probs`` are inverse-CDF
    quantiles (hist_quantiles); ``counts`` holds the pooled histograms and ``n_samples`` the pooled sample count."""
    run = batch.run
    ranges = run.cfg.store >= STORE_FULL
    m = run.marginals(np.asarray(chains, dtype=np.int32), ranges=ranges)
    pooled = {key: (m[key].sum(axis=0, dtype=np.int64).astype(np.int32) if m[key] is not None else None) for key in ("pos", "a", "b")}
    return dict(sites=_marginal_summary(pooled["pos"], probs),
                a=_marginal_summary(pooled["a"], probs) if ranges else None,
                b=_marginal_summary(pooled["b"], probs) if ranges else None,
                counts=pooled, n_samples=int(m["n_samples"].sum()), probs=tuple(probs))


def compute_exp_cd(batch: ChainBatch, chains, chains_selected: int, faithful: bool = True):
    """script.py:102-126: per chosen chain the sum over its samples of exp(c), exp(d) divided by the LITERAL 1000
    (:119-120; like compute_exp_ages / _pi / _a and exp_data.csv -- equal to the mean only for the reference's
    1000 samples), summed over the chains and divided by ``chains_selected``.  ``faithful=False`` divides by the
    number of samples actually taken."""
    st = batch.stats()
    scale = st["n_samples"] / 1000 if faithful else 1.0
    return (float(np.sum(st["e_c"][list(chains)]) * scale / chains_selected),
            float(np.sum(st["e_d"][list(chains)]) * scale / chains_selected))


def pearson_from_corr_num(corr_num, n_samples: int, n_sites: int):
    """mean over samples of pearsonr(pi_t, arange(N)) from sum_t sum_i i*pi_t(i): pi_t is a permutation of
    0..N-1, so both series have mean (N-1)/2 and variance (N^2-1)/12"""
    N = float(n_sites)
    mean, var = (N - 1.0) / 2.0, (N * N - 1.0) / 12.0
    return (np.asarray(corr_num, dtype=np.float64) / (n_samples * N) - mean * mean) / var


def carry_over_mean(per_chain_sums, chains_selected: int, keep_total: bool, faithful: bool = True):
    """The accumulation pattern of compute_exp_pi / compute_exp_a (script.py:230-276): the per-chain
    accumulator is divided by 1000 but never reset, so chain c starts from chain c-1's scaled values
    (``faithful``); compute_exp_a adds every chain's accumulator into the total (``keep_total``), while
    compute_exp_pi resets the total inside the loop (:243), so only the LAST chain's accumulator survives."""
    carry = np.zeros_like(np.asarray(per_chain_sums[0], dtype=np.float64))
    total = np.zeros_like(carry)
    for sums in per_chain_sums:
        acc = ((carry if faithful else 0.0) + np.asarray(sums, dtype=np.float64)) / 1000
        total = total + acc if (keep_total or not faithful) else acc
        carry = acc
    return total / chains_selected


def compute_exp_ages(batch: ChainBatch, chains, chains_selected: int, sites: int | None = None):
    """script.py:129-152: expected Pearson correlation of pi with the file order, per-chain means (divided by the
    literal 1000) summed over the chosen chains and divided by ``chains_selected``."""
    ps = batch.run.posterior_sums(np.asarray(chains, dtype=np.int32))
    r = pearson_from_corr_num(ps["corr_num"], ps["n_samples"], batch.run.N)   # mean over the T stored samples
    return float(np.sum(r * ps["n_samples"] / 1000) / chains_selected)


def compute_exp_pi(batch: ChainBatch, chains, sites: int | None, chains_selected: int, faithful: bool = True):
    """script.py:230-252 (with its reset/carry-over quirks when ``faithful``)"""
    ps = batch.run.posterior_sums(np.asarray(chains, dtype=np.int32))
    return carry_over_mean(list(ps["pi_sum"]), chains_selected, keep_total=False, faithful=faithful)


def compute_exp_a(batch: ChainBatch, chains, chains_selected: int, taxa: int | None = None, faithful: bool = True):
    """script.py:255-276; needs a batch created with the full sample store"""
    ps = batch.run.posterior_sums(np.asarray(chains, dtype=np.int32), with_ab=True)
    return carry_over_mean(list(ps["a_sum"]), chains_selected, keep_total=True, faithful=faithful)


def _reorder_like_script(X_sum, exp_pi, exp_a):
    """script.py:339-353: row r <- the row at site r's rank in exp_pi; column i <- taxon argsort(exp_a)[i]"""
    rpi = np.argsort(exp_pi)
    idx = np.empty_like(rpi)
    idx[rpi] = np.arange(len(rpi))
    return X_sum[idx, :][:, np.argsort(exp_a)]


def _interval_map(batch: ChainBatch, chains, chains_selected: int, cell, faithful: bool):
    alive, T = batch.run.alive_counts(np.asarray(chains, dtype=np.int32))
    X_sum = carry_over_mean([cell(alive[c].astype(np.float64), T) for c in range(len(alive))], chains_selected,
                            keep_total=True, faithful=faithful)
    return _reorder_like_script(X_sum, compute_exp_pi(batch, chains, None, chains_selected, faithful),
                                compute_exp_a(batch, chains, chains_selected, None, faithful))


def taxa_occurence_probability_matrix(batch: ChainBatch, chains, chains_selected: int, sites: int | None = None,
                                      taxa: int | None = None, faithful: bool = True):
    """What plot_taxa_occurence_probability_matrix returns (script.py:306-353): X_ij = Pr(taxon i alive at
    position j), rows ordered by E[pi], columns by E[a]; interval closed at b as the reference tests it;
    counts on the GPU (ser_run_alive_counts).  Needs a batch with the full sample store."""
    return _interval_map(batch, chains, chains_selected, lambda alive, T: alive, faithful)


def false_taxa_occurence_probability_matrix(batch: ChainBatch, chains, chains_selected: int, sites: int | None = None,
                                            taxa: int | None = None, faithful: bool = True):
    """plot_false_taxa_occurence_probability's matrix (script.py:356-403): Pr(taxon i not alive at j)"""
    return _interval_map(batch, chains, chains_selected, lambda alive, T: T - alive, faithful)


def false_ones_probability_matrix(batch: ChainBatch, chains, chains_selected: int, dataset=None, sites: int | None = None,
                                  taxa: int | None = None, faithful: bool = True):
    """plot_false_ones_probability's matrix (script.py:406-448): Pr(X_ij = 1 is a false one).  The reference
    indexes X by FILE row while a, b are positions; kept.  ``dataset``: path / Dataset, default the batch's own."""
    ds = batch.run.ds if dataset is None else (dataset if isinstance(dataset, Dataset) else Dataset.read_txt(str(dataset)))
    X = ds.arrays()[0].astype(np.float64)
    return _interval_map(batch, chains, chains_selected, lambda alive, T: X * (T - alive), faithful)


def new_data_matrix(batch: ChainBatch, chains, chains_selected: int, dataset=None, sites: int | None = None,
                    taxa: int | None = None, faithful: bool = True):
    """The matrix plot_new_data_matrix draws (script.py:279-303): occurrences with sites ordered by E[pi]
    and taxa by E[a]."""
    ds = batch.run.ds if dataset is None else (dataset if isinstance(dataset, Dataset) else Dataset.read_txt(str(dataset)))
    return _reorder_like_script(ds.arrays()[0].astype(np.float64), compute_exp_pi(batch, chains, None, chains_selected, faithful),
                                compute_exp_a(batch, chains, chains_selected, None, faithful))
