"""The pairwise-error / NDCG@k evaluation (util.cpp:434-542) against the CPU oracle, user by user, and the read-only entry
points of the stage API against the training trajectory they must not change.

Three kernels evaluate (csrc/k_pairs.cu): eval_pairs (all-pairs error count), eval_users (top-k by repeated arg-max, one
warp per user) and eval_sorted<T> (error count and NDCG from the Primal-CR++ sorted state, instantiated for T <= 5 and
T <= 8 levels).  Every one is compared with oracle.eval_scores on the same scores, at every ndcg_k class (1, around the
default 10, around a warp, up to the limit 64), at rows shorter than, equal to and one longer than ndcg_k, and with the
planted ties of test_gpu_kernel_classes (integer runs across 32-lane chunks, float32-colliding runs, +-1e39).

Bars: per-user pair-error counts identical; per-user NDCG within 1e-13 relative (CUDA exp2 / log2 against libm);
all-pairs and sorted-state per-user NDCG bit-identical to each other; means within 1e-12; NaN where the oracle has NaN.
"""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import bindings as ob
from primalcr_b200 import api
from primalcr_b200.data import Dataset, Ratings, csr_in_file_order
from tests.test_gpu_kernel_classes import int_inputs, plant_p1, plant_p2, plant_p3, size_dataset
from tests.test_gpu_parity import VEC_TOL, check_sorted_state
from tests.util import dataset, init_factors, np_init, rel, to_csr

gpu = pytest.mark.gpu

NDCG_K = [1, 2, 9, 10, 11, 31, 32, 33, 63, 64]
EXTRA_LENS = [3, 9, 10, 11, 31, 32, 33, 62, 63, 64, 65]      # rows around every ndcg_k boundary, on top of size_dataset
PLANTS = dict(P1=(plant_p1, NDCG_K), P2=(plant_p2, [1, 10, 64]), P3=(plant_p3, [1, 10, 64]))
T_LIST = [2, 5, 6, 8, 9, 12]


def engine(ds, ndcg_k, solver=2, U=None, V=None, levels=True, k=None):
    """make_engine with a given ndcg_k (fixed when an engine is created)."""
    k = k if k is not None else (U.shape[1] if U is not None else 5)
    e = api.Engine(api.Parameter(solver_type=solver, k=k, lambda_=4.0, maxiter=3, ndcg_k=ndcg_k))
    if levels is True:
        levels = np.unique(np.rint(ds.train.rating).astype(np.int64))
    if levels is not None and levels is not False:
        e.set_levels(levels)
    e.set_train(ds.train)
    if ds.test.nnz:
        e.set_test(ds.test)
    if U is None:
        U, V, _, _ = int_inputs(ds.d1, ds.d2, k, seed=17)
    e.set_factors(U, V)
    return e


def got_eval(e, which, method):
    err, nd, cnt, ndu = e.eval_error_counts(which, method, ndcg_per_user=True)
    return np.array([err, nd]), cnt, ndu


def assert_eval(got, want, what):
    """got: (means, per-user counts, per-user NDCG) from the engine; want: oracle.eval_scores / eval(per_user=True)."""
    means, cnt, ndu = got
    wmeans, _, wcnt, wndu = want
    assert np.array_equal(cnt, wcnt), (what, np.flatnonzero(cnt != wcnt)[:10])
    nan = np.isnan(wndu)
    assert np.array_equal(np.isnan(ndu), nan), (what, np.flatnonzero(np.isnan(ndu) != nan)[:10])
    bad = np.flatnonzero(np.abs(ndu[~nan] - wndu[~nan]) > 1e-13 * np.abs(wndu[~nan]))
    assert bad.size == 0, (what, np.flatnonzero(~nan)[bad[:10]], ndu[~nan][bad[:10]], wndu[~nan][bad[:10]])
    for g, w in zip(means, wmeans):
        assert (np.isnan(g) and np.isnan(w)) or abs(g - w) <= 1e-12, (what, means, wmeans)


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


# ----------------------------------------------------------------------------- 1. the oracle's new entry point (CPU)
@pytest.mark.parametrize("name", ["tiny", "ragged", "ragged_real"])
def test_oracle_eval_scores_matches_eval(name):
    """eval_scores on comp_m(U, V) is eval at (U, V): counts, per-user values and means bit for bit."""
    ds = dataset(name)
    O = ob.oracle()
    U, V = np_init(ds.d1, ds.d2, 6, seed=31, scale=0.7)
    V[1::5] = V[0]                                  # exact score ties
    U[3] = 0.0                                      # a user whose scores all tie at 0
    for R in (ds.train, ds.test):
        X = to_csr(R)
        for k in (1, 10, 64):
            want = O.eval(X, U, V, k, per_user=True)
            got = O.eval_scores(X, O.comp_m(X, U, V), k)
            assert same_bits(got[0], want[0]) and np.array_equal(got[1], want[1])
            assert np.array_equal(got[2], want[2]) and same_bits(got[3], want[3])
            assert same_bits(want[0], O.eval(X, U, V, k))
            assert np.array_equal(want[2], O.eval(X, U, V, k, want_counts=True)[2])
            # the mean NDCG is the in-order average of the per-user values over the non-empty rows
            ne = np.diff(R.row_ptr) > 0
            s = 0.0
            for x in want[3][ne]:
                s += x
            assert same_bits(s / ne.sum(), want[0][1]) and not want[3][~ne].any()


# ----------------------------------------------------------------------------- 2. planted scores x level tables
_cache = {}


def eval_dataset(T):
    """size_dataset(T) (rows of 0 ... 16385 ratings) plus rows of EXTRA_LENS ratings, integer ratings 1..T."""
    if T not in _cache:
        base = size_dataset(T).train
        rng = np.random.default_rng(200 + T)
        us, its, vs = [base.users()], [base.item], [base.rating]
        for q, n in enumerate(EXTRA_LENS):
            us.append(np.full(n, base.d1 + q)); its.append(rng.choice(base.d2, n, replace=False))
            vs.append(rng.integers(1, T + 1, n).astype(np.float64))
        d1 = base.d1 + len(EXTRA_LENS)
        R = Ratings.from_coo(d1, base.d2, np.concatenate(us), np.concatenate(its), np.concatenate(vs))
        _cache[T] = Dataset(R, Ratings.empty(d1, base.d2), name="eval_T%d" % T)
    return _cache[T]


def oracle_planted(T):
    """oracle.eval_scores of every (plant, ndcg_k) of eval_dataset(T), computed on all cores (the oracle call releases
    the GIL; its O(len^2) loop over the 16385-rating row dominates)."""
    key = ("oracle", T)
    if key not in _cache:
        R = eval_dataset(T).train
        X = to_csr(R)
        O = ob.oracle()
        scores = {p: f(R, T) for p, (f, _) in PLANTS.items()}
        jobs = [(p, k) for p, (_, ks) in PLANTS.items() for k in ks]
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
            res = list(ex.map(lambda j: O.eval_scores(X, scores[j[0]], j[1]), jobs))
        _cache[key] = (scores, dict(zip(jobs, res)))
    return _cache[key]


def test_eval_dataset_premise():
    """The rows this module relies on are there: every ndcg_k class has rows shorter, equal and one longer."""
    for T in (2, 12):
        lens = np.diff(eval_dataset(T).train.row_ptr)
        assert lens.max() == 16385 and 0 in lens
        for k in NDCG_K:
            assert {k - 1, k, k + 1} - {0} <= set(lens.tolist()), k
        assert set(np.unique(eval_dataset(T).train.rating)) == set(range(1, T + 1))


def sorted_kernel(T):
    return "eval_sorted_T5" if T <= 5 else "eval_sorted_T8"


@gpu
@pytest.mark.parametrize("T", T_LIST)
def test_planted_scores_all_kernels(T):
    ds = eval_dataset(T)
    scores, want = oracle_planted(T)
    for k in NDCG_K:
        e = engine(ds, k)
        assert e.num_levels() == T
        e.profile_enable(True)
        for p, (_, ks) in PLANTS.items():
            if k not in ks:
                continue
            what = (T, p, k)
            e.set_scores(scores[p])
            e.profile_reset()
            g0 = got_eval(e, 0, 0)
            prof = {n for n, v in e.profile().items() if v["launches"] > 0}
            assert {"eval_pairs", "eval_users"} <= prof and not any(n.startswith("eval_sorted") for n in prof), prof
            assert_eval(g0, want[(p, k)], what + (0,))
            if T <= 8:
                e.profile_reset()
                g1 = got_eval(e, 0, 1)
                prof = {n for n, v in e.profile().items() if v["launches"] > 0}
                assert sorted_kernel(T) in prof and "eval_pairs" not in prof and "eval_users" not in prof, prof
                assert_eval(g1, want[(p, k)], what + (1,))
                assert np.array_equal(g1[1], g0[1]) and same_bits(g1[2], g0[2]) and same_bits(g1[0], g0[0]), what
            else:
                with pytest.raises(api.PrimalCRError, match="<= 8 levels"):
                    e.eval_error_counts(0, method=1)
                e.profile_reset()
                assert same_bits(e.eval(0), g0[0]), what
                prof = {n for n, v in e.profile().items() if v["launches"] > 0}
                assert {"eval_pairs", "eval_users"} <= prof and not any(n.startswith("eval_sorted") for n in prof)
        e.close()


# ----------------------------------------------------------------------------- 3. level-table edges
def small_dataset(seed, values, lens=(0, 1, 2, 3, 9, 10, 11, 31, 32, 33, 40, 63, 64, 65, 100, 300, 1100, 5000),
                  all_zero_user=False, d2=6000):
    rng = np.random.default_rng(seed)
    us, its, vs = [], [], []
    for u, n in enumerate(lens):
        us.append(np.full(n, u)); its.append(rng.choice(d2, n, replace=False))
        vs.append(rng.choice(np.asarray(values, np.float64), n))
    if all_zero_user:
        vs[5][:] = 0.0
    d1 = len(lens)
    R = Ratings.from_coo(d1, d2, np.concatenate(us), np.concatenate(its), np.concatenate(vs))
    return Dataset(R, Ratings.empty(d1, d2), name="levels")


def tie_scores(R, seed):
    """Integer scores in [-3, 3] with -0.0 next to +0.0: ties everywhere, runs longer than a 32-lane chunk."""
    rng = np.random.default_rng(seed)
    m = rng.integers(-3, 4, R.nnz).astype(np.float64)
    z = np.flatnonzero(m == 0.0)
    m[z[::2]] = -0.0
    return m


@gpu
def test_level_table_one_and_eight():
    """Ratings {1, 8}: the library's lo..hi table (T = 8, six empty levels) and set_levels([1, 8]) (T = 2) give the same
    per-user results as each other and as the oracle."""
    ds = small_dataset(1, [1, 8])
    m = tie_scores(ds.train, 1)
    X = to_csr(ds.train)
    for k in (1, 10, 33, 64):
        want = ob.oracle().eval_scores(X, m, k)
        got = {}
        for T, levels in ((8, None), (2, [1, 8])):
            e = engine(ds, k, levels=levels)
            assert e.num_levels() == T
            e.set_scores(m)
            e.profile_enable(True)
            for method in (0, 1):
                got[(T, method)] = got_eval(e, 0, method)
                assert_eval(got[(T, method)], want, (k, T, method))
            assert "eval_sorted_T5" in e.profile() if T == 2 else "eval_sorted_T8" in e.profile()
            e.close()
        ref = got[(8, 0)]
        for g in got.values():
            assert same_bits(g[0], ref[0]) and np.array_equal(g[1], ref[1]) and same_bits(g[2], ref[2]), k


@gpu
def test_zero_gains_and_nan_ndcg():
    """Ratings 0..7 (a gain of 0 for rating 0; T = 8) and a user whose ratings are all 0: its ideal DCG is 0, so its NDCG
    -- and the mean -- are NaN in the engine as in the oracle."""
    ds = small_dataset(2, np.arange(8), all_zero_user=True)
    m = tie_scores(ds.train, 2)
    X = to_csr(ds.train)
    for k in (1, 10, 64):
        want = ob.oracle().eval_scores(X, m, k)
        assert np.isnan(want[3][5]) and np.isnan(want[0][1]) and np.isfinite(want[3][np.arange(len(want[3])) != 5]).all()
        e = engine(ds, k)
        assert e.num_levels() == 8
        e.set_scores(m)
        g0, g1 = got_eval(e, 0, 0), got_eval(e, 0, 1)
        assert_eval(g0, want, (k, 0)); assert_eval(g1, want, (k, 1))
        assert same_bits(g0[2], g1[2])
        e.close()


@gpu
def test_no_comparable_pair_is_nan():
    """Every user has at most one rating: no pair anywhere, the pairwise error is 0 / 0 = NaN in both; NDCG is 1."""
    ds = small_dataset(3, [1, 2, 3, 4, 5], lens=(0, 1, 1, 0, 1, 1, 1, 0))
    m = tie_scores(ds.train, 3)
    want = ob.oracle().eval_scores(to_csr(ds.train), m, 10)
    assert np.isnan(want[0][0]) and want[0][1] == 1.0
    e = engine(ds, 10)
    e.set_scores(m)
    for method in (0, 1):
        g = got_eval(e, 0, method)
        assert_eval(g, want, method)
        assert np.isnan(g[0][0])
    e.close()


# ----------------------------------------------------------------------------- 4. test set: long rows, exact ties
TEST_LENS = [0, 1, 2, 31, 32, 33, 255, 256, 257, 1023, 1024, 1025, 2049, 5000]


def long_rows_dataset():
    """A few training ratings per user; test rows of TEST_LENS entries in file order, repeated items in some rows."""
    if "test_set" not in _cache:
        rng = np.random.default_rng(9)
        d2 = 6000
        d1 = len(TEST_LENS)
        us, its, vs, tu, ti, tv = [], [], [], [], [], []
        for u, n in enumerate(TEST_LENS):
            us.append(np.full(4, u)); its.append(rng.choice(d2, 4, replace=False)); vs.append(rng.integers(1, 6, 4) * 1.0)
            tu.append(np.full(n, u)); ti.append(rng.choice(d2, n, replace=(u % 3 == 1)))
            tv.append(rng.integers(1, 6, n).astype(np.float64))
        train = Ratings.from_coo(d1, d2, np.concatenate(us), np.concatenate(its), np.concatenate(vs))
        test = csr_in_file_order(d1, d2, np.concatenate(tu), np.concatenate(ti), np.concatenate(tv))
        _cache["test_set"] = Dataset(train, test, name="long_test_rows")
    return _cache["test_set"]


@gpu
@pytest.mark.parametrize("factors", ["integer", "real"])
def test_long_test_rows(factors):
    """eval_error_counts(1, 0) on test rows of up to 5000 entries (several 256-entry pair work items and 1024-entry
    shared-memory stages per user) against oracle.eval per user, at every ndcg_k.  Integer factors in {-1, 0, 1} with
    k = 2 put every score in {-2..2}: long exact tie runs."""
    ds = long_rows_dataset()
    T = ds.test
    assert any(len(np.unique(T.item[T.row_ptr[u]:T.row_ptr[u + 1]])) < n for u, n in enumerate(TEST_LENS))
    if factors == "integer":
        U, V, _, _ = int_inputs(ds.d1, ds.d2, 2, seed=5)
    else:
        U, V = np_init(ds.d1, ds.d2, 2, seed=5, scale=0.8)
    X = to_csr(T)
    O = ob.oracle()
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        want = dict(zip(NDCG_K, ex.map(lambda k: O.eval(X, U, V, k, per_user=True), NDCG_K)))
    for k in NDCG_K:
        e = engine(ds, k, U=U, V=V)
        assert_eval(got_eval(e, 1, 0), want[k], k)
        assert same_bits(e.eval(1), got_eval(e, 1, 0)[0])
        e.close()


# ----------------------------------------------------------------------------- 5. Primal-CR and the driver
@gpu
def test_pcr_engine_evaluation():
    """Primal-CR (-s 1) evaluates with the all-pairs kernels, the same numbers; it has no sorted state to use."""
    T = 5
    ds = eval_dataset(T)
    scores, want = oracle_planted(T)
    for k in (1, 10, 64):
        e = engine(ds, k, solver=1)
        e.set_scores(scores["P1"])
        assert_eval(got_eval(e, 0, 0), want[("P1", k)], k)
        with pytest.raises(api.PrimalCRError, match="Primal-CR\\+\\+"):
            e.eval_error_counts(0, method=1)
        e.close()


@gpu
@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("ndcg_k", [1, 33, 64])
def test_driver_ndcg_k(solver, ndcg_k):
    """pcrpp() / pcr() with do_predict = 1 and a non-default ndcg_k: the banner names it, and every (Training) / (Testing)
    line carries the oracle's numbers to the printed precision."""
    ds = dataset("ragged")
    k, lam, iters = 10, 20.0, 2
    U, V = init_factors(ds.d1, ds.d2, k)
    res = ob.oracle().train(solver, to_csr(ds.train), to_csr(ds.test), U, V, lam, iters, do_predict=1, ndcg_k=ndcg_k)
    p = api.Parameter(solver_type=solver, k=k, lambda_=lam, maxiter=iters, do_predict=1, ndcg_k=ndcg_k)
    lines = (api.pcrpp if solver == 2 else api.pcr)(ds.train, U.copy(), V.copy(), ds.test, p, log=None)
    assert lines[0] == ("running PrimalCR++ ndcg_k is %d" if solver == 2 else "running PrimalCR ndcg_k is %d") % ndcg_k
    tr = [l.split() for l in lines if l.startswith("(Training)")]
    te = [l.split() for l in lines if l.startswith("(Testing)")]
    assert len(tr) == iters + 1 and len(te) == iters + 1
    for i in range(iters + 1):
        for got, want in ((tr[i][4], res["evals"][i, 0]), (tr[i][-1], res["evals"][i, 1]),
                          (te[i][4], res["evals"][i, 2]), (te[i][-1], res["evals"][i, 3])):
            assert abs(float(got) - want) <= 5e-6 * abs(want) + 1e-15, (i, got, want)


# ----------------------------------------------------------------------------- 6. read-only calls leave training alone
STEPSIZES = [1.0, 48.0, 1.0e6]      # 1e6: the first V line search rejects all 20 trials
READS = ["eval0", "eval1", "counts0", "counts1", "counts0_sorted", "objective", "grad_V", "hv_V", "grad_U", "hv_U",
         "sort_segments", "level_counts", "scores", "get_factors", "counters"]
SOLVER2_ONLY = {"counts0_sorted", "sort_segments", "level_counts"}
RO_K, RO_LAM = 7, 50.0


def ro_engine(solver, stepsize):
    ds = dataset("tiny")
    U, V = init_factors(ds.d1, ds.d2, RO_K)
    e = api.Engine(api.Parameter(solver_type=solver, k=RO_K, lambda_=RO_LAM, maxiter=3, stepsize=stepsize))
    e.set_levels(np.unique(np.rint(ds.train.rating).astype(np.int64)))
    e.set_train(ds.train); e.set_test(ds.test); e.set_factors(U, V)
    return e


def ro_run(solver, stepsize, read=None, check=None):
    """Three outer iterations through the stage API; `read` is called between update_V and update_U and after update_U.
    Returns everything observable after each half step: objective, the eight counters, both factors."""
    e = ro_engine(solver, stepsize)
    out = []
    for _ in range(3):
        for step in (e.update_V, e.update_U):
            o = step()
            c = e.counters()
            Ug, Vg = e.get_factors()
            out.append((o, c, Ug, Vg))
            if read is not None:
                r = do_read(e, read, solver)
                if check is not None:
                    check(read, r, solver, (o, c, Ug, Vg))
    e.close()
    return out


_dirs = {}


def directions():
    if not _dirs:
        ds = dataset("tiny")
        rng = np.random.default_rng(77)
        _dirs.update(a=rng.standard_normal((ds.d2, RO_K)), S=rng.standard_normal((ds.d1, RO_K)))
    return _dirs


def do_read(e, read, solver):
    d = directions()
    if read == "eval0": return e.eval(0)
    if read == "eval1": return e.eval(1)
    if read == "counts0": return got_eval(e, 0, 0)
    if read == "counts1": return got_eval(e, 1, 0)
    if read == "counts0_sorted": return got_eval(e, 0, 1)
    if read == "objective": return e.objective()
    if read == "grad_V": return e.grad_V()
    if read == "hv_V": return e.hv_V(d["a"])
    if read == "grad_U": return e.grad_U()
    if read == "hv_U": return e.hv_U(d["S"])
    if read == "sort_segments": return e.sort_segments()
    if read == "level_counts": return e.sort_segments(), e.level_counts()
    if read == "scores": return e.scores()
    if read == "get_factors": return e.get_factors()
    if read == "counters": return e.counters()
    raise AssertionError(read)


def check_read(read, r, solver, state):
    """A read's own result against the oracle at the current factors (or against the state just recorded)."""
    _, c, U, V = state
    ds = dataset("tiny")
    O = ob.oracle()
    X = to_csr(ds.train)
    m = O.comp_m(X, U, V)
    if read in ("eval0", "eval1"):
        R = ds.train if read == "eval0" else ds.test
        w = O.eval(to_csr(R), U, V, 10)
        assert abs(r[0] - w[0]) <= 1e-12 and abs(r[1] - w[1]) <= 1e-12, (read, r, w)
    elif read.startswith("counts"):
        R = ds.test if read == "counts1" else ds.train
        assert_eval(r, O.eval(to_csr(R), U, V, 10, per_user=True), read)
    elif read == "objective":
        w = O.objective_new(X, m, U, V, RO_LAM) if solver == 2 else O.pcr_objective(X, m, U, V, RO_LAM)
        assert abs(r - w) <= 1e-12 * abs(w), (r, w)
    elif read == "grad_V":
        assert rel(r, O.obtain_g_new(X, U, V, m, RO_LAM) if solver == 2 else O.pcr_obtain_g(X, U, V, m, RO_LAM)) < VEC_TOL
    elif read == "hv_V":
        a = directions()["a"]
        assert rel(r, O.compute_Ha_new(X, a, m, U, RO_LAM) if solver == 2 else O.pcr_compute_Ha(X, a, m, U, RO_LAM)) < VEC_TOL
    elif read in ("grad_U", "hv_U") and solver == 2:
        rp = ds.train.row_ptr
        S = directions()["S"]
        w = [O.user_stage(X.rows[rp[u]:rp[u + 1]], X.vals[rp[u]:rp[u + 1]], m[rp[u]:rp[u + 1]], V, RO_LAM, U[u], S[u])
             for u in range(ds.d1)]
        if read == "grad_U":          # relative to the largest entry: a converged user's gradient is rounding noise
            assert rel(r[0], np.array([x[0] for x in w])) < VEC_TOL
            oo = np.array([x[1] for x in w])
            assert np.all(np.abs(r[1] - oo) <= 1e-12 * np.maximum(np.abs(oo), 1.0))
        else:
            has = np.diff(rp) > 0
            assert rel(r[has], np.array([x[2] for x in w])[has]) < VEC_TOL
    elif read in ("sort_segments", "level_counts"):
        out = r if read == "sort_segments" else r[0]
        mg = np.empty(ds.train.nnz)                 # the engine's scores, put back in CSR order by its permutation
        rp = ds.train.row_ptr
        for u in range(ds.d1):
            a, b = int(rp[u]), int(rp[u + 1])
            mg[a + out["perm"][a:b]] = out["sorted"][a:b]
        assert rel(mg, m) < 1e-13
        if read == "level_counts":
            check_sorted_state(ds.train, mg, out, *r[1], np.unique(np.rint(ds.train.rating).astype(np.int64)))
    elif read == "scores":
        assert rel(r, m) < 1e-13
    elif read == "get_factors":
        assert np.array_equal(r[0], U) and np.array_equal(r[1], V)
    elif read == "counters":
        assert r == c


_base = {}


def baseline(solver, stepsize):
    if (solver, stepsize) not in _base:
        _base[(solver, stepsize)] = ro_run(solver, stepsize)
    return _base[(solver, stepsize)]


@gpu
@pytest.mark.parametrize("solver,stepsize,read", [(s, st, r) for s in (2, 1) for st in STEPSIZES for r in READS
                                                  if s == 2 or r not in SOLVER2_ONLY])
def test_read_only_calls_do_not_change_training(solver, stepsize, read):
    """Calling a read-only entry point between update_V and update_U, and after update_U, leaves every objective, counter
    and factor of three outer iterations bit-identical -- in particular after a V line search that rejected all its
    trials, whose last trial's scores update_U consumes (pcrpp.cpp:443) -- and returns the oracle's value itself."""
    want = baseline(solver, stepsize)
    assert any(s[1]["v_ls_accepted"] == 0 for s in want) == (stepsize > 1e3)
    got = ro_run(solver, stepsize, read, check_read)
    for i, (g, w) in enumerate(zip(got, want)):
        assert same_bits(g[0], w[0]), (i, g[0], w[0])
        assert g[1] == w[1], (i, g[1], w[1])
        assert same_bits(g[2], w[2]) and same_bits(g[3], w[3]), i
