"""ctypes bindings for the parity oracle -- TEST INFRASTRUCTURE ONLY.

Two libraries, same argument conventions (flat numpy arrays, CSR by user with int64 indices):
  * ``liboracle.so``        -- plain-C restatement (oracle/pcr_oracle.c), always buildable with gcc;
  * ``_ref/libref_harness.so`` -- the UNMODIFIED reference objects behind oracle/ref_harness.cpp,
    present only where /root/reference was available at build time (it then travels with gpurun).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
Nothing under primalcr_b200/ does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_P = np.ctypeslib.ndpointer
_f64 = _P(dtype=np.float64, flags="C_CONTIGUOUS")
_i64 = _P(dtype=np.int64, flags="C_CONTIGUOUS")
_l, _d, _i = C.c_long, C.c_double, C.c_int


def build(ref: bool = True) -> None:
    """Compile liboracle.so (and oracle/_ref when /root/reference exists)."""
    targets = ["oracle"] + (["ref"] if ref else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True)


def _load(path):
    return C.CDLL(path) if os.path.exists(path) else None


def _opt(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Csr:
    """CSR by user with the reference's SparseMat field meanings (util.h:390-413)."""

    def __init__(self, d1, d2, index, rows, vals):
        self.d1, self.d2 = int(d1), int(d2)
        self.index = np.ascontiguousarray(index, dtype=np.int64)
        self.rows = np.ascontiguousarray(rows, dtype=np.int64)
        self.vals = np.ascontiguousarray(vals, dtype=np.float64)
        self.nnz = int(self.index[-1])
        assert len(self.index) == self.d1 + 1 and len(self.rows) >= self.nnz

    def args(self):
        return (self.d1, self.d2, self.nnz, self.index, self.rows, self.vals)

    @staticmethod
    def empty(d1, d2):
        return Csr(d1, d2, np.zeros(d1 + 1, np.int64), np.zeros(1, np.int64), np.zeros(1, np.float64))


class _Lib:
    """Common wrapper: `prefix` is 'orc_' for the C restatement, 'ref_' for the reference harness."""

    def __init__(self, lib, prefix):
        self.lib, self.prefix = lib, prefix
        csr = [_l, _l, _l, _i64, _i64, _f64]
        g = lambda name: getattr(lib, prefix + name)
        f = g("comp_m"); f.restype = None
        f.argtypes = ([_l, _l, _l, _i64, _i64] + ([_f64] if prefix == "ref_" else [])) + [_f64, _f64, _i, _f64]
        f = g("sorted_mm"); f.restype = None; f.argtypes = [_f64, _l, _f64, _i64]
        f = g("obtain_g_new"); f.restype = None; f.argtypes = csr + [_f64, _f64, _i, _f64, _d, _f64]
        f = g("compute_Ha_new"); f.restype = None; f.argtypes = csr + [_f64, _f64, _f64, _i, _d, _f64]
        f = g("objective_new"); f.restype = _d; f.argtypes = csr + [_f64, _f64, _f64, _i, _d]
        f = g("eval"); f.restype = None
        f.argtypes = csr + [_f64, _f64, _i, _i, _f64] + ([C.c_void_p, C.c_void_p, C.c_void_p] if prefix == "orc_" else [])
        if prefix == "orc_":
            f = g("eval_scores"); f.restype = None
            f.argtypes = [_l, _i64, _f64, _f64, _i, _f64, _i64, _i64, _f64]
        f = g("pcr_obtain_g"); f.restype = None
        f = g("pcr_compute_Ha"); f.restype = None
        f = g("pcr_objective"); f.restype = _d
        if prefix == "orc_":
            g("pcr_objective").argtypes = [_l, _l, _i64, _f64, _f64, _f64, _f64, _i, _d]
            g("pcr_obtain_g").argtypes = [_l, _l, _i64, _i64, _f64, _f64, _f64, _i, _f64, _d, _f64]
            g("pcr_compute_Ha").argtypes = [_l, _l, _i64, _i64, _f64, _f64, _f64, _f64, _i, _d, _f64]
        else:
            g("pcr_objective").argtypes = csr + [_f64, _f64, _f64, _i, _d]
            g("pcr_obtain_g").argtypes = csr + [_f64, _f64, _i, _f64, _d, _f64]
            g("pcr_compute_Ha").argtypes = csr + [_f64, _f64, _f64, _i, _d, _f64]
        f = g("user_stage"); f.restype = None
        if prefix == "orc_":
            f.argtypes = [_l, _i64, _f64, _f64, _f64, _i, _d, _f64, _f64, _f64, _f64, _f64]
        else:
            f.argtypes = [_l, _i64, _f64, _f64, _f64, _l, _i, _d, _f64, _f64, _f64, _f64, _f64]
        f = g("train"); f.restype = None
        f.argtypes = [_i] + csr + [_l, _i64, _i64, _f64, _f64, _f64, _i, _d, _d, _i, _i, _i] + \
            ([_f64, C.c_void_p, C.c_void_p] if prefix == "orc_" else [_i, _f64, C.c_void_p])

    # ---- stage functions -------------------------------------------------
    def comp_m(self, X, U, V):
        r = U.shape[1]
        m = np.zeros(max(X.nnz, 1))
        if self.prefix == "ref_":
            self.lib.ref_comp_m(*X.args(), U, V, r, m)
        else:
            self.lib.orc_comp_m(X.d1, X.d2, X.nnz, X.index, X.rows, U, V, r, m)
        return m[:X.nnz]

    def sorted_mm(self, mm):
        mm = np.ascontiguousarray(mm, dtype=np.float64)
        s = np.zeros(max(len(mm), 1)); p = np.zeros(max(len(mm), 1), np.int64)
        getattr(self.lib, self.prefix + "sorted_mm")(mm if len(mm) else np.zeros(1), len(mm), s, p)
        return s[:len(mm)], p[:len(mm)]

    def obtain_g_new(self, X, U, V, m, lam):
        g = np.zeros_like(V)
        getattr(self.lib, self.prefix + "obtain_g_new")(*X.args(), U, V, U.shape[1], _pad(m), lam, g)
        return g

    def compute_Ha_new(self, X, a, m, U, lam):
        Ha = np.zeros_like(a)
        getattr(self.lib, self.prefix + "compute_Ha_new")(*X.args(), a, _pad(m), U, U.shape[1], lam, Ha)
        return Ha

    def objective_new(self, X, m, U, V, lam):
        return getattr(self.lib, self.prefix + "objective_new")(*X.args(), _pad(m), U, V, U.shape[1], lam)

    def pcr_objective(self, X, m, U, V, lam):
        if self.prefix == "orc_":
            return self.lib.orc_pcr_objective(X.d1, X.d2, X.index, X.vals, _pad(m), U, V, U.shape[1], lam)
        return self.lib.ref_pcr_objective(*X.args(), _pad(m), U, V, U.shape[1], lam)

    def pcr_obtain_g(self, X, U, V, m, lam):
        g = np.zeros_like(V)
        if self.prefix == "orc_":
            self.lib.orc_pcr_obtain_g(X.d1, X.d2, X.index, X.rows, X.vals, U, V, U.shape[1], _pad(m), lam, g)
        else:
            self.lib.ref_pcr_obtain_g(*X.args(), U, V, U.shape[1], _pad(m), lam, g)
        return g

    def pcr_compute_Ha(self, X, a, m, U, lam):
        Ha = np.zeros_like(a)
        if self.prefix == "orc_":
            self.lib.orc_pcr_compute_Ha(X.d1, X.d2, X.index, X.rows, X.vals, a, _pad(m), U, U.shape[1], lam, Ha)
        else:
            self.lib.ref_pcr_compute_Ha(*X.args(), a, _pad(m), U, U.shape[1], lam, Ha)
        return Ha

    def user_stage(self, rows, vals, m, V, lam, ui, s):
        """(g_u, objective_u, Hs) of one user: obtain_g_u_new / objective_u_new / obtain_Hs_new."""
        r = V.shape[1]
        n = len(rows)
        rows = np.ascontiguousarray(rows, np.int64); vals = np.ascontiguousarray(vals, np.float64)
        g = np.zeros(r); Hs = np.zeros(r); obj = np.zeros(1)
        if self.prefix == "orc_":
            self.lib.orc_user_stage(n, _padl(rows), _pad(vals), _pad(m), V, r, lam, ui, s, g, obj, Hs)
        else:
            self.lib.ref_user_stage(n, _padl(rows), _pad(vals), _pad(m), V, V.shape[0], r, lam, ui, s, g, obj, Hs)
        return g, float(obj[0]), Hs

    def eval(self, X, U, V, ndcg_k=10, want_counts=False, per_user=False):
        """[pairwise error, ndcg]; want_counts: (that, the 4 totals, per-user error counts); per_user: the same plus the
        per-user NDCG (NaN where the ideal DCG is 0, 0 for an empty row)."""
        out = np.zeros(2)
        if self.prefix == "orc_":
            counts = np.zeros(4, np.int64); err = np.zeros(max(X.d1, 1), np.int64); nd = np.zeros(max(X.d1, 1))
            self.lib.orc_eval(*X.args(), U, V, U.shape[1], ndcg_k, out, _opt(counts), _opt(err), _opt(nd))
            if per_user:
                return out, counts, err[:X.d1], nd[:X.d1]
            if want_counts:
                return out, counts, err[:X.d1]
        else:
            assert not (want_counts or per_user), "the reference harness returns the two means only"
            self.lib.ref_eval(*X.args(), U, V, U.shape[1], ndcg_k, out)
        return out

    def eval_scores(self, X, m, ndcg_k=10):
        """eval() from given scores m (one per rating of X, CSR order): (means, 4 totals, per-user error counts,
        per-user NDCG)."""
        assert self.prefix == "orc_"
        m = np.ascontiguousarray(m, np.float64)
        assert len(m) == X.nnz
        out = np.zeros(2); counts = np.zeros(4, np.int64)
        err = np.zeros(max(X.d1, 1), np.int64); nd = np.zeros(max(X.d1, 1))
        self.lib.orc_eval_scores(X.d1, X.index, X.vals, _pad(m), ndcg_k, out, counts, err, nd)
        return out, counts, err[:X.d1], nd[:X.d1]

    def train(self, solver, X, XT, U, V, lam, maxiter, do_predict=1, ndcg_k=10, stepsize=1.0, threads=1):
        """Runs `maxiter` outer iterations; returns dict(obj, evals, U, V[, counters])."""
        U = np.array(U, dtype=np.float64, order="C"); V = np.array(V, dtype=np.float64, order="C")
        if XT is None:
            XT = Csr.empty(X.d1, X.d2)
        obj = np.zeros(maxiter + 1); evals = np.zeros((maxiter + 1, 4))
        res = dict(obj=obj, evals=evals, U=U, V=V)
        base = (solver,) + X.args() + (XT.nnz, XT.index, XT.rows, XT.vals, U, V, U.shape[1], lam, stepsize,
                                       maxiter, do_predict, ndcg_k)
        if self.prefix == "orc_":
            counters = np.zeros((max(maxiter, 1), 8), np.int64)
            self.lib.orc_train(*base, obj, _opt(evals), _opt(counters))
            res["counters"] = counters[:maxiter]
        else:
            self.lib.ref_train(*base, threads, obj, _opt(evals))
        return res


def _pad(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a if a.size else np.zeros(1)


def _padl(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a if a.size else np.zeros(1, np.int64)


_orc = _ref = None


def oracle() -> _Lib:
    """The plain-C restatement (built on demand)."""
    global _orc
    if _orc is None:
        path = os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(os.path.join(HERE, "pcr_oracle.c")):
            build(ref=False)
        lib = C.CDLL(path)
        lib.orc_level_counts.restype = None
        lib.orc_level_counts.argtypes = [_f64, _f64, _l, _i64, _f64, _i64, _i64, _i64, _i64]
        lib.orc_update_V_new.restype = None
        lib.orc_update_U_new.restype = None
        _orc = _Lib(lib, "orc_")
    return _orc


def reference():
    """The unmodified reference behind the harness, or None when oracle/_ref was never built."""
    global _ref
    if _ref is None:
        lib = _load(os.path.join(HERE, "_ref", "libref_harness.so"))
        if lib is None:
            return None
        lib.ref_initial.restype = None
        lib.ref_initial.argtypes = [_f64, _l, _l]
        _ref = _Lib(lib, "ref_")
    return _ref


_ref_rf = None


def reference_rf():
    """The reference harness over the race-free objects (obj_u_new made loop-local, see oracle/Makefile): the build to use
    with threads > 1.  None when oracle/_ref was never built."""
    global _ref_rf
    if _ref_rf is None:
        lib = _load(os.path.join(HERE, "_ref", "libref_harness_rf.so"))
        if lib is None:
            return None
        _ref_rf = _Lib(lib, "ref_")
    return _ref_rf


def ref_initial(n, k):
    out = np.zeros((n, k))
    reference().lib.ref_initial(out, n, k)
    return out


def level_counts(mm, vals):
    """Per-position window counters of one user (the loop locals of pcrpp.cpp:206-229)."""
    lib = oracle().lib
    n = len(mm)
    mm = _pad(mm); vals = _pad(vals)
    nl = np.zeros(1, np.int64)
    s = np.zeros(max(n, 1)); perm = np.zeros(max(n, 1), np.int64); lev = np.zeros(max(n, 1), np.int64)
    tmax = max(len(np.unique(np.rint(vals[:n]))) if n else 1, 1)
    cl = np.zeros(max(n, 1) * tmax, np.int64); cr = np.zeros(max(n, 1) * tmax, np.int64)
    lib.orc_level_counts(mm, vals, n, nl, s, perm, lev, cl, cr)
    T = int(nl[0])
    return dict(T=T, s=s[:n], perm=perm[:n], level=lev[:n], cntL=cl[:n * T].reshape(n, T) if T else cl[:0].reshape(n, 0),
                cntR=cr[:n * T].reshape(n, T) if T else cr[:0].reshape(n, 0))


def ref_cli(name="omp-pmf-train"):
    p = os.path.join(HERE, "_ref", name)
    return p if os.path.exists(p) else None
