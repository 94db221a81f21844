"""Python host side above the C ABI (include/primalcr.h).

Mirrors the reference's solver interface for this path (pmf.h:9-56): a ``Parameter`` object with the same
field names and defaults as ``class parameter``, and ``pcr(X, U, V, T, param)`` / ``pcrpp(X, U, V, T, param)``
that update U and V in place and print the reference's log lines.  Everything numerical happens in
``libprimalcr_b200.so`` (hand-written sm_100a kernels); if the library or a GPU is missing the calls raise
-- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

from .data import Ratings

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PRIMALCR_LIB") or os.path.join(_HERE, "libprimalcr_b200.so")   # PRIMALCR_LIB: A/B builds

CCDR1, PCR, PCRPP = 0, 1, 2   # pmf.h:6


class PrimalCRError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [("solver", C.c_int), ("k", C.c_int), ("lambda_", C.c_double), ("stepsize", C.c_double),
                ("maxiter", C.c_int), ("ndcg_k", C.c_int), ("do_predict", C.c_int), ("device", C.c_int),
                ("threads", C.c_int)]


class Counters(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("v_cg_iters", "v_ls_trials", "v_ls_accepted", "u_cg_len_sum",
                                         "u_ls_len_sum", "u_skipped", "u_cg_iters", "u_ls_trials")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


# every symbol include/primalcr.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "primalcr_default_config", "primalcr_create", "primalcr_destroy", "primalcr_last_error", "primalcr_version",
    "primalcr_set_levels", "primalcr_set_train_csr", "primalcr_set_test_csr", "primalcr_set_factors",
    "primalcr_get_factors", "primalcr_nccl_unique_id", "primalcr_comm_init", "primalcr_initial_objective",
    "primalcr_update_V", "primalcr_update_U", "primalcr_outer_iteration", "primalcr_eval", "primalcr_eval_error_counts",
    "primalcr_run",
    "primalcr_get_counters", "primalcr_scores", "primalcr_set_scores", "primalcr_sort_segments",
    "primalcr_level_counts", "primalcr_num_levels", "primalcr_objective", "primalcr_grad_V", "primalcr_hv_V",
    "primalcr_grad_U", "primalcr_hv_U", "primalcr_stream", "primalcr_launch_count", "primalcr_profile_enable",
    "primalcr_profile_reset", "primalcr_profile_count", "primalcr_profile_get", "primalcr_device_bytes",
    "primalcr_reference_init", "primalcr_write_text_matrix", "primalcr_predict", "primalcr_load_dir", "primalcr_dataset_info",
    "primalcr_dataset_csr", "primalcr_dataset_free", "primalcr_recommend", "primalcr_rank_heldout", "primalcr_rank_metrics",
]

_lib = None
LOG_FN = C.CFUNCTYPE(None, C.c_char_p, C.c_void_p)


def build_library(force: bool = False) -> str:
    """nvcc build of csrc/ for sm_100a into primalcr_b200/libprimalcr_b200.so (in-tree)."""
    src = os.path.join(_HERE, "csrc")
    if force:
        subprocess.run(["make", "-s", "-C", src, "clean"], check=True)
    subprocess.run(["make", "-s", "-j8", "-C", src], check=True)
    return LIB_PATH


def lib():
    """Loads libprimalcr_b200.so; raises when it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PrimalCRError("libprimalcr_b200.so is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                            "or `make -C primalcr_b200/csrc` -- there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32p, i64p, f64p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
    L.primalcr_last_error.restype = C.c_char_p
    L.primalcr_version.restype = C.c_char_p
    L.primalcr_default_config.argtypes = [C.POINTER(_Config)]
    L.primalcr_create.argtypes = [C.POINTER(vp), C.POINTER(_Config)]
    L.primalcr_destroy.argtypes = [vp]; L.primalcr_destroy.restype = None
    L.primalcr_set_levels.argtypes = [vp, i64p, C.c_int]
    L.primalcr_set_train_csr.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, i64p, i32p, f64p]
    L.primalcr_set_test_csr.argtypes = [vp, C.c_int64, i64p, i32p, f64p]
    L.primalcr_set_factors.argtypes = [vp, f64p, f64p]
    L.primalcr_get_factors.argtypes = [vp, f64p, f64p]
    L.primalcr_nccl_unique_id.argtypes = [vp]
    L.primalcr_comm_init.argtypes = [vp, C.c_int, C.c_int, vp]
    for name in ("initial_objective", "objective", "update_V", "update_U", "outer_iteration"):
        getattr(L, "primalcr_" + name).argtypes = [vp, C.POINTER(C.c_double)]
    L.primalcr_eval.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.primalcr_eval_error_counts.argtypes = [vp, C.c_int, C.c_int, vp, vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.primalcr_run.argtypes = [vp, LOG_FN, vp]
    L.primalcr_get_counters.argtypes = [vp, C.POINTER(Counters)]
    L.primalcr_scores.argtypes = [vp, f64p]
    L.primalcr_set_scores.argtypes = [vp, f64p]
    L.primalcr_sort_segments.argtypes = [vp, f64p, i32p, i32p, i32p, i32p, i32p, i32p]
    L.primalcr_level_counts.argtypes = [vp, i32p, i32p]
    L.primalcr_num_levels.argtypes = [vp]
    L.primalcr_grad_V.argtypes = [vp, f64p]
    L.primalcr_hv_V.argtypes = [vp, f64p, f64p]
    L.primalcr_grad_U.argtypes = [vp, f64p, f64p]
    L.primalcr_hv_U.argtypes = [vp, f64p, f64p]
    L.primalcr_stream.argtypes = [vp]; L.primalcr_stream.restype = vp
    L.primalcr_launch_count.argtypes = [vp]; L.primalcr_launch_count.restype = C.c_int64
    L.primalcr_profile_enable.argtypes = [vp, C.c_int]
    L.primalcr_profile_reset.argtypes = [vp]
    L.primalcr_profile_count.argtypes = [vp]
    L.primalcr_profile_get.argtypes = [vp, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double),
                                       C.POINTER(C.c_int64), C.POINTER(C.c_double)]
    L.primalcr_device_bytes.argtypes = [vp]; L.primalcr_device_bytes.restype = C.c_int64
    L.primalcr_reference_init.argtypes = [f64p, C.c_int64, C.c_int64]; L.primalcr_reference_init.restype = None
    L.primalcr_write_text_matrix.argtypes = [C.c_char_p, f64p, C.c_int64, C.c_int]
    L.primalcr_predict.argtypes = [f64p, C.c_int64, f64p, C.c_int64, C.c_int, i32p, i32p, C.c_int64, f64p, C.c_int]
    L.primalcr_recommend.argtypes = [f64p, C.c_int64, f64p, C.c_int64, C.c_int, i64p, i32p, i32p, C.c_int64, C.c_int, i32p,
                                     f64p, C.c_int]
    L.primalcr_rank_heldout.argtypes = [f64p, C.c_int64, f64p, C.c_int64, C.c_int, i64p, i32p, i64p, i32p, i32p, f64p, C.c_int]
    L.primalcr_rank_metrics.argtypes = [C.c_int64, C.c_int64, i64p, i32p, i64p, i32p, f64p, i32p, C.c_double, i32p, C.c_int,
                                        f64p, f64p, f64p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                        C.POINTER(C.c_int64)]
    L.primalcr_load_dir.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    L.primalcr_dataset_info.argtypes = [vp] + [C.POINTER(C.c_int64)] * 4
    L.primalcr_dataset_csr.argtypes = [vp, C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    L.primalcr_dataset_free.argtypes = [vp]; L.primalcr_dataset_free.restype = None
    _lib = L
    return L


def _ptr(a):
    """Address of a numpy array / torch CPU tensor / None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()   # torch tensor (pinned host memory in bench.py)


def _require_factor(a, rows: int, k: int, name: str):
    """The C ABI reads / writes rows*k doubles through a raw pointer: insist on a C-contiguous float64 (rows, k) buffer."""
    if isinstance(a, np.ndarray):
        ok = a.dtype == np.float64 and a.flags.c_contiguous and a.flags.writeable and a.shape == (rows, k)
    else:       # torch CPU tensor
        import torch
        ok = isinstance(a, torch.Tensor) and a.dtype == torch.float64 and a.device.type == "cpu" and a.is_contiguous() \
            and tuple(a.shape) == (rows, k)
    if not ok:
        raise PrimalCRError("%s must be a C-contiguous float64 array of shape (%d, %d), got %s %s" % (
            name, rows, k, getattr(a, "dtype", type(a)), tuple(getattr(a, "shape", ()))))


def reference_init(n: int, k: int) -> np.ndarray:
    """initial() util.cpp:80-93 -- the default-seeded N(0,1) stream of the reference CLI (host code, libstdc++)."""
    out = np.empty((n, k), np.float64)
    lib().primalcr_reference_init(out.ctypes.data, n, k)
    return out


def write_text_matrix(path: str, M: np.ndarray) -> None:
    """U.txt / V.txt as the reference CLI writes them (pmf-train.cpp:276-295), formatted in parallel on the host."""
    M = np.ascontiguousarray(M, np.float64)
    rc = lib().primalcr_write_text_matrix(path.encode(), M.ctypes.data, M.shape[0], M.shape[1])
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))


def load_dir(path: str, threads: int = 0):
    """The library's parallel mmap loader for a reference data directory (host/loader.hpp) -> data.Dataset."""
    from .data import Dataset
    L = lib()
    h = C.c_void_p()
    rc = L.primalcr_load_dir(path.encode(), threads, C.byref(h))
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, L.primalcr_last_error().decode()))
    try:
        d1, d2, n0, n1 = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        L.primalcr_dataset_info(h, C.byref(d1), C.byref(d2), C.byref(n0), C.byref(n1))
        out = []
        for which, n in ((0, n0.value), (1, n1.value)):
            rp, it, ra = C.c_void_p(), C.c_void_p(), C.c_void_p()
            L.primalcr_dataset_csr(h, which, C.byref(rp), C.byref(it), C.byref(ra))
            row_ptr = np.ctypeslib.as_array(C.cast(rp, C.POINTER(C.c_int64)), (d1.value + 1,)).copy()
            item = np.ctypeslib.as_array(C.cast(it, C.POINTER(C.c_int32)), (n,)).copy() if n else np.zeros(0, np.int32)
            rating = np.ctypeslib.as_array(C.cast(ra, C.POINTER(C.c_double)), (n,)).copy() if n else np.zeros(0)
            out.append(Ratings(d1.value, d2.value, row_ptr, item, rating))
        return Dataset(out[0], out[1], name=os.path.basename(os.path.normpath(path)))
    finally:
        L.primalcr_dataset_free(h)


def predict(U, V, users, items, device: int = 0) -> np.ndarray:
    """omp-pmf-predict's loop (pmf-predict.cpp:57-64) as one GPU batch: out[t] = U[users[t]] . V[items[t]] (0-based)."""
    U = np.ascontiguousarray(U, np.float64); V = np.ascontiguousarray(V, np.float64)
    users = np.ascontiguousarray(users, np.int32); items = np.ascontiguousarray(items, np.int32)
    out = np.empty(len(users))
    rc = lib().primalcr_predict(U.ctypes.data, U.shape[0], V.ctypes.data, V.shape[0], U.shape[1], users.ctypes.data,
                                items.ctypes.data, len(users), out.ctypes.data, device)
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))
    return out


def recommend(U, V, n: int, exclude: Ratings | None = None, users=None, device: int = 0):
    """Top-n items of every requested user by U[u] . V[i] over all items, skipping the user's items in `exclude`
    (normally the training set) -> (items int32 (n_users, n), scores float64 (n_users, n)).

    Rows are sorted best first, ties to the smaller item id, NaN scores last; a user with fewer than n eligible items is
    padded with item -1 / score NaN.  users: 0-based ids in any order, repeats allowed (default: every user)."""
    U = np.ascontiguousarray(U, np.float64); V = np.ascontiguousarray(V, np.float64)
    if U.ndim != 2 or V.ndim != 2 or U.shape[1] != V.shape[1]:
        raise PrimalCRError("U and V must be 2-D with the same number of columns, got %s and %s" % (U.shape, V.shape))
    d1, d2, k = U.shape[0], V.shape[0], U.shape[1]
    rp = it = None
    if exclude is not None:
        if exclude.d1 != d1 or exclude.d2 != d2:
            raise PrimalCRError("exclude is %d x %d, the factors are %d x %d" % (exclude.d1, exclude.d2, d1, d2))
        rp = np.ascontiguousarray(exclude.row_ptr, np.int64); it = np.ascontiguousarray(exclude.item, np.int32)
        if len(rp) != d1 + 1 or len(it) < rp[-1]:
            raise PrimalCRError("exclude: row_ptr needs d1+1 entries and item row_ptr[d1]")
    if users is not None:
        users = np.ascontiguousarray(users, np.int32).reshape(-1)
    n_users = d1 if users is None else len(users)
    items = np.empty((n_users, max(int(n), 0)), np.int32)
    scores = np.empty((n_users, max(int(n), 0)), np.float64)
    rc = lib().primalcr_recommend(U.ctypes.data, d1, V.ctypes.data, d2, k, _ptr(rp), _ptr(it), _ptr(users), n_users,
                                  int(n), items.ctypes.data, scores.ctypes.data, device)
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))
    return items, scores


def _csr_arrays(R: Ratings, d1: int, d2: int, name: str):
    """(row_ptr int64, item int32) of a d1 x d2 Ratings, checked for the lengths the C ABI reads."""
    if R.d1 != d1 or R.d2 != d2:
        raise PrimalCRError("%s is %d x %d, expected %d x %d" % (name, R.d1, R.d2, d1, d2))
    rp = np.ascontiguousarray(R.row_ptr, np.int64); it = np.ascontiguousarray(R.item, np.int32)
    if len(rp) != d1 + 1 or len(it) < rp[-1]:
        raise PrimalCRError("%s: row_ptr needs d1+1 entries and item row_ptr[d1]" % name)
    return rp, it


def heldout_ranks(U, V, heldout: Ratings, exclude: Ratings | None = None, device: int = 0):
    """The catalog rank of every held-out entry -> (ranks int32 [nnz], scores float64 [nnz]), in heldout's CSR order.

    rank = 1 + the number of the user's items outside `exclude` (normally the training set) that api.recommend would put
    before the entry's item; 0 when the item itself is excluded.  So an entry of rank r <= n is at position r-1 of
    api.recommend(U, V, n, exclude)'s row for that user, with the same score bit for bit."""
    U = np.ascontiguousarray(U, np.float64); V = np.ascontiguousarray(V, np.float64)
    if U.ndim != 2 or V.ndim != 2 or U.shape[1] != V.shape[1]:
        raise PrimalCRError("U and V must be 2-D with the same number of columns, got %s and %s" % (U.shape, V.shape))
    d1, d2, k = U.shape[0], V.shape[0], U.shape[1]
    hp, hi = _csr_arrays(heldout, d1, d2, "heldout")
    rp = it = None
    if exclude is not None:
        rp, it = _csr_arrays(exclude, d1, d2, "exclude")
    nnz = int(hp[-1])
    ranks = np.empty(max(nnz, 0), np.int32); scores = np.empty(max(nnz, 0), np.float64)
    rc = lib().primalcr_rank_heldout(U.ctypes.data, d1, V.ctypes.data, d2, k, _ptr(rp), _ptr(it), hp.ctypes.data,
                                     hi.ctypes.data, ranks.ctypes.data, scores.ctypes.data, device)
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))
    return ranks, scores


def ranking_metrics(ranks, heldout: Ratings, exclude: Ratings | None = None, cutoffs=(10,), min_rating=None) -> dict:
    """recall@N, precision@N, ndcg@N for every N in cutoffs, mrr, auc and n_users from heldout_ranks' ranks (host only).

    A held-out item is relevant when its rating is >= min_rating (None: every item); the definitions are those of
    primalcr_rank_metrics in include/primalcr.h.  `exclude` must be the one the ranks were computed with."""
    d1, d2 = heldout.d1, heldout.d2
    hp, hi = _csr_arrays(heldout, d1, d2, "heldout")
    hr = np.ascontiguousarray(heldout.rating, np.float64)
    ranks = np.ascontiguousarray(ranks, np.int32).reshape(-1)
    if len(ranks) < hp[-1] or len(hr) < hp[-1]:
        raise PrimalCRError("ranks and heldout.rating need heldout.row_ptr[d1] entries")
    rp = it = None
    if exclude is not None:
        rp, it = _csr_arrays(exclude, d1, d2, "exclude")
    cuts = np.ascontiguousarray(cutoffs, np.int32).reshape(-1)
    nc = len(cuts)
    rec, prec, ndcg = np.empty(nc), np.empty(nc), np.empty(nc)
    mrr, auc, n_users = C.c_double(), C.c_double(), C.c_int64()
    rc = lib().primalcr_rank_metrics(d1, d2, _ptr(rp), _ptr(it), hp.ctypes.data, hi.ctypes.data, hr.ctypes.data,
                                     ranks.ctypes.data, -np.inf if min_rating is None else float(min_rating),
                                     cuts.ctypes.data, nc, rec.ctypes.data, prec.ctypes.data, ndcg.ctypes.data,
                                     C.byref(mrr), C.byref(auc), C.byref(n_users))
    if rc != 0:
        raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))
    out = {}
    for j, n in enumerate(cuts):
        out["recall@%d" % n] = float(rec[j]); out["precision@%d" % n] = float(prec[j]); out["ndcg@%d" % n] = float(ndcg[j])
    out.update(mrr=mrr.value, auc=auc.value, n_users=int(n_users.value))
    return out


@dataclass
class Parameter:
    """``class parameter`` pmf.h:9-49 (the fields pcr()/pcrpp() read), same names and defaults."""
    solver_type: int = PCRPP
    k: int = 10
    threads: int = 4          # echoed in the "using N threads. " log line only; has no meaning on the GPU
    maxiter: int = 10
    lambda_: float = 5000.0   # `lambda` in the reference
    stepsize: float = 1.0
    ndcg_k: int = 10
    do_predict: int = 1
    verbose: int = 0
    device: int = 0


class Engine:
    """One GPU's share of the training path.  Thin, explicit wrapper: one method per C-ABI entry point."""

    def __init__(self, param: Parameter, solver: int | None = None):
        L = lib()
        cfg = _Config()
        L.primalcr_default_config(C.byref(cfg))
        cfg.solver = int(solver if solver is not None else param.solver_type)
        cfg.k = int(param.k); cfg.lambda_ = float(param.lambda_); cfg.stepsize = float(param.stepsize)
        cfg.maxiter = int(param.maxiter); cfg.ndcg_k = int(param.ndcg_k); cfg.do_predict = int(param.do_predict)
        cfg.device = int(param.device); cfg.threads = int(param.threads)
        self.k = cfg.k
        self._h = C.c_void_p()
        self._L = L
        self._check(L.primalcr_create(C.byref(self._h), C.byref(cfg)))
        self.d1 = self.d2 = self.nnz = 0
        self._keep = []

    def _check(self, rc):
        if rc != 0:
            raise PrimalCRError("primalcr error %d: %s" % (rc, self._L.primalcr_last_error().decode()))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.primalcr_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- data
    def set_levels(self, values):
        v = np.ascontiguousarray(values, np.int64)
        self._check(self._L.primalcr_set_levels(self._h, v.ctypes.data, len(v)))

    def set_train(self, R: Ratings):
        rp = np.ascontiguousarray(R.row_ptr, np.int64)
        self.set_train_raw(R.d1, R.d2, R.nnz, rp, np.ascontiguousarray(R.item, np.int32),
                           np.ascontiguousarray(R.rating, np.float64))

    def set_train_raw(self, d1, d2, nnz, row_ptr, item, rating):
        """row_ptr/item/rating: numpy arrays or (pinned) torch CPU tensors of int64/int32/float64."""
        self._check(self._L.primalcr_set_train_csr(self._h, d1, d2, nnz, _ptr(row_ptr), _ptr(item), _ptr(rating)))
        self.d1, self.d2, self.nnz = int(d1), int(d2), int(nnz)

    def set_test(self, R: Ratings):
        rp = np.ascontiguousarray(R.row_ptr, np.int64)
        it = np.ascontiguousarray(R.item, np.int32); ra = np.ascontiguousarray(R.rating, np.float64)
        self._check(self._L.primalcr_set_test_csr(self._h, R.nnz, rp.ctypes.data, it.ctypes.data, ra.ctypes.data))
        self.nnz_test = R.nnz

    def set_factors(self, U, V):
        if isinstance(U, np.ndarray):
            U = np.ascontiguousarray(U, np.float64); V = np.ascontiguousarray(V, np.float64)
        _require_factor(U, self.d1, self.k, "U"); _require_factor(V, self.d2, self.k, "V")
        self._check(self._L.primalcr_set_factors(self._h, _ptr(U), _ptr(V)))

    def get_factors(self, U=None, V=None):
        """Writes d1*k and d2*k doubles through the raw pointers of U and V: both must be C-contiguous float64
        (d1, k) / (d2, k) buffers (numpy arrays or torch CPU tensors); anything else raises instead of corrupting memory."""
        if U is None:
            U = np.empty((self.d1, self.k)); V = np.empty((self.d2, self.k))
        _require_factor(U, self.d1, self.k, "U"); _require_factor(V, self.d2, self.k, "V")
        self._check(self._L.primalcr_get_factors(self._h, _ptr(U), _ptr(V)))
        return U, V

    # ---- multi-GPU
    @staticmethod
    def nccl_unique_id() -> bytes:
        buf = C.create_string_buffer(128)
        rc = lib().primalcr_nccl_unique_id(buf)
        if rc != 0:
            raise PrimalCRError("primalcr error %d: %s" % (rc, lib().primalcr_last_error().decode()))
        return buf.raw

    def comm_init(self, rank: int, world: int, uid: bytes | None):
        buf = C.create_string_buffer(uid, 128) if uid is not None else None
        self._check(self._L.primalcr_comm_init(self._h, rank, world, buf))

    # ---- solver
    def _scalar(self, fn):
        v = C.c_double()
        self._check(fn(self._h, C.byref(v)))
        return v.value

    def initial_objective(self): return self._scalar(self._L.primalcr_initial_objective)
    def objective(self): return self._scalar(self._L.primalcr_objective)
    def update_V(self): return self._scalar(self._L.primalcr_update_V)
    def update_U(self): return self._scalar(self._L.primalcr_update_U)
    def outer_iteration(self): return self._scalar(self._L.primalcr_outer_iteration)

    def eval(self, which: int = 0):
        a, b = C.c_double(), C.c_double()
        self._check(self._L.primalcr_eval(self._h, which, C.byref(a), C.byref(b)))
        return a.value, b.value

    def eval_error_counts(self, which: int = 0, method: int = 0, ndcg_per_user: bool = False):
        """(pairwise error, NDCG, integer pair-error count per user[, NDCG per user]); method 0 all pairs, 1 sorted state
        (Primal-CR++ train set).  A user's NDCG is 0 for an empty row and NaN when its ideal DCG is 0."""
        n = self.d1
        cnt = np.zeros(max(n, 1), np.int64)
        nd = np.zeros(max(n, 1)) if ndcg_per_user else None
        a, b = C.c_double(), C.c_double()
        self._check(self._L.primalcr_eval_error_counts(self._h, which, method, cnt.ctypes.data,
                                                       None if nd is None else nd.ctypes.data, C.byref(a), C.byref(b)))
        if ndcg_per_user:
            return a.value, b.value, cnt[:n], nd[:n]
        return a.value, b.value, cnt[:n]

    def run(self, log=print):
        lines = []
        def _cb(line, _ctx):
            s = line.decode()
            lines.append(s)
            if log is not None:
                log(s)
        cb = LOG_FN(_cb)
        self._check(self._L.primalcr_run(self._h, cb, None))
        return lines

    def counters(self) -> dict:
        c = Counters()
        self._check(self._L.primalcr_get_counters(self._h, C.byref(c)))
        return c.as_dict()

    # ---- stages
    def scores(self):
        m = np.empty(max(self.nnz, 1))
        self._check(self._L.primalcr_scores(self._h, m.ctypes.data))
        return m[:self.nnz]

    def set_scores(self, m):
        m = np.ascontiguousarray(m, np.float64)
        self._check(self._L.primalcr_set_scores(self._h, m.ctypes.data if m.size else None))

    def num_levels(self): return int(self._L.primalcr_num_levels(self._h))

    def sort_segments(self):
        n = max(self.nnz, 1)
        out = dict(sorted=np.empty(n), perm=np.empty(n, np.int32), level=np.empty(n, np.int32),
                   ub=np.empty(n, np.int32), lb=np.empty(n, np.int32), cnt_lo=np.empty(n, np.int32),
                   cnt_hi=np.empty(n, np.int32))
        self._check(self._L.primalcr_sort_segments(self._h, *[out[k].ctypes.data for k in
                                                              ("sorted", "perm", "level", "ub", "lb", "cnt_lo", "cnt_hi")]))
        return {k: v[:self.nnz] for k, v in out.items()}

    def level_counts(self):
        T = self.num_levels()
        cl = np.empty((max(self.nnz, 1), T), np.int32); cr = np.empty((max(self.nnz, 1), T), np.int32)
        self._check(self._L.primalcr_level_counts(self._h, cl.ctypes.data, cr.ctypes.data))
        return cl[:self.nnz], cr[:self.nnz]

    def grad_V(self):
        g = np.empty((self.d2, self.k))
        self._check(self._L.primalcr_grad_V(self._h, g.ctypes.data))
        return g

    def hv_V(self, a):
        a = np.ascontiguousarray(a, np.float64).reshape(self.d2, self.k)
        out = np.empty((self.d2, self.k))
        self._check(self._L.primalcr_hv_V(self._h, a.ctypes.data, out.ctypes.data))
        return out

    def grad_U(self):
        g = np.empty((self.d1, self.k)); o = np.empty(max(self.d1, 1))
        self._check(self._L.primalcr_grad_U(self._h, g.ctypes.data, o.ctypes.data))
        return g, o[:self.d1]

    def hv_U(self, S):
        S = np.ascontiguousarray(S, np.float64).reshape(self.d1, self.k)
        out = np.empty((self.d1, self.k))
        self._check(self._L.primalcr_hv_U(self._h, S.ctypes.data, out.ctypes.data))
        return out

    # ---- measurement
    def stream_ptr(self) -> int: return int(self._L.primalcr_stream(self._h) or 0)
    def launch_count(self) -> int: return int(self._L.primalcr_launch_count(self._h))
    def device_bytes(self) -> int: return int(self._L.primalcr_device_bytes(self._h))
    def profile_enable(self, on=True): self._check(self._L.primalcr_profile_enable(self._h, 1 if on else 0))
    def profile_reset(self): self._check(self._L.primalcr_profile_reset(self._h))

    def profile(self) -> dict:
        out = {}
        for i in range(self._L.primalcr_profile_count(self._h)):
            name = C.c_char_p(); ms = C.c_double(); n = C.c_int64(); b = C.c_double()
            self._check(self._L.primalcr_profile_get(self._h, i, C.byref(name), C.byref(ms), C.byref(n), C.byref(b)))
            out[name.value.decode()] = dict(ms=ms.value, launches=n.value, bytes=b.value)
        return out


# ----------------------------------------------------------------------------- the reference's solver interface

def _solve(solver, X: Ratings, U: np.ndarray, V: np.ndarray, T: Ratings | None, param: Parameter, log=print):
    _require_factor(U, X.d1, param.k, "U"); _require_factor(V, X.d2, param.k, "V")     # in/out buffers: checked before any work
    eng = Engine(param, solver=solver)
    try:
        eng.set_train(X)
        if T is not None and T.nnz:
            eng.set_test(T)
        eng.set_factors(U, V)
        lines = eng.run(log)
        eng.get_factors(U, V)     # in/out, like the reference's mat_t& U, mat_t& V
        return lines
    finally:
        eng.close()


def pcrpp(X: Ratings, U: np.ndarray, V: np.ndarray, T: Ratings | None, param: Parameter, log=print):
    """Drop-in for ``pcrpp(smat_t&, mat_t& U, mat_t& V, testset_t&, parameter&)`` pmf.h:55 / pcrpp.cpp:841."""
    return _solve(PCRPP, X, U, V, T, param, log)


def pcr(X: Ratings, U: np.ndarray, V: np.ndarray, T: Ratings | None, param: Parameter, log=print):
    """Drop-in for ``pcr(smat_t&, mat_t& U, mat_t& V, testset_t&, parameter&)`` pmf.h:54 / pcr.cpp:616."""
    return _solve(PCR, X, U, V, T, param, log)
