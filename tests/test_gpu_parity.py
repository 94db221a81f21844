"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): sorted orders and per-level window counts bit-exact given identical scores;
objective per outer iteration within 1e-6 relative (we assert 1e-9); test NDCG@10 within 1e-4; the integer
control-flow counters (CG iterations, line-search trials, skipped users) identical.
"""
import numpy as np
import pytest

from oracle import bindings as ob
from primalcr_b200 import api
from tests.util import dataset, init_factors, np_init, rel, to_csr

pytestmark = pytest.mark.gpu

OBJ_TOL = 1e-9      # north_star allows 1e-6 relative
NDCG_TOL = 1e-4     # north_star
VEC_TOL = 1e-9      # gradients / Hv / factors: relative to the largest entry


def make_engine(ds, k, lam, solver=2, U=None, V=None, test=True, maxiter=3, levels=True):
    p = api.Parameter(solver_type=solver, k=k, lambda_=lam, maxiter=maxiter)
    e = api.Engine(p)
    if levels:
        vals = np.unique(np.rint(ds.train.rating).astype(np.int64))
        e.set_levels(vals)
    e.set_train(ds.train)
    if test and ds.test.nnz:
        e.set_test(ds.test)
    if U is None:
        U, V = init_factors(ds.d1, ds.d2, k)
    e.set_factors(U, V)
    return e, U, V


@pytest.mark.parametrize("name,k", [("tiny", 7), ("ragged", 10), ("ragged", 100), ("tiny", 200)])
def test_scores(name, k):
    ds = dataset(name)
    e, U, V = make_engine(ds, k, 50.0)
    m = e.scores()
    mo = ob.oracle().comp_m(to_csr(ds.train), U, V)
    assert rel(m, mo) < 1e-13
    e.close()


def check_sorted_state(R, m, out, cl, cr, levels):
    """The engine's sorted state (sort_segments() -> out, level_counts() -> cl, cr) of every user of R under the scores m
    against the oracle's, bit for bit.  levels: the engine's global level table."""
    rp = R.row_ptr
    for u in range(R.d1):
        a, b = int(rp[u]), int(rp[u + 1])
        if a == b:
            continue
        o = ob.level_counts(m[a:b], R.rating[a:b])
        assert np.array_equal(out["sorted"][a:b].view(np.int64), o["s"].view(np.int64)), u   # bit pattern, -0.0 != +0.0
        # permutation: valid, and equal to the oracle's wherever the key is unique
        perm = out["perm"][a:b]
        assert np.array_equal(np.sort(perm), np.arange(b - a))
        assert np.array_equal(m[a:b][perm], o["s"])
        assert np.array_equal(perm, o["perm"]), u          # both break ties by index
        # levels: oracle's are user-local ranks, ours global ranks
        lv_user = np.unique(np.rint(R.rating[a:b]).astype(np.int64))
        glob = np.searchsorted(levels, lv_user)
        assert np.array_equal(out["level"][a:b], glob[o["level"]])
        # window pointers and per-level counters (loop locals of pcrpp.cpp:206-229)
        assert np.array_equal(out["ub"][a:b], o["cntL"].sum(1)), u
        assert np.array_equal((b - a) - out["lb"][a:b], o["cntR"].sum(1)), u
        assert np.array_equal(cl[a:b][:, glob], o["cntL"]), u
        assert np.array_equal(cr[a:b][:, glob], o["cntR"]), u
        other = np.setdiff1d(np.arange(len(levels)), glob)
        assert not cl[a:b][:, other].any() and not cr[a:b][:, other].any()
        lev = o["level"]
        col = np.arange(o["cntL"].shape[1])[None, :]
        hi = np.where(col > lev[:, None], o["cntL"], 0).sum(1)
        lo = np.where(col < lev[:, None], o["cntR"], 0).sum(1)
        assert np.array_equal(out["cnt_hi"][a:b], hi), u
        assert np.array_equal(out["cnt_lo"][a:b], lo), u


@pytest.mark.parametrize("name", ["tiny", "ragged", "ragged_real"])
def test_sort_and_counts_bitexact(name):
    """Identical scores in -> identical sorted order, window pointers and per-level counters out."""
    ds = dataset(name)
    k = 6
    U, V = np_init(ds.d1, ds.d2, k, seed=11, scale=0.6)
    X = to_csr(ds.train)
    m = ob.oracle().comp_m(X, U, V)
    # plant exact ties and +-0.0 inside a few users
    rp = ds.train.row_ptr
    for u in range(ds.d1):
        a, b = int(rp[u]), int(rp[u + 1])
        if b - a >= 6:
            m[a + 1] = m[a + 4]; m[a + 2] = 0.0; m[a + 3] = -0.0; m[a + 5] = m[a + 4] + 1.0
    e, _, _ = make_engine(ds, k, 50.0, U=U, V=V)
    e.set_scores(m)
    out = e.sort_segments()
    cl, cr = e.level_counts()
    check_sorted_state(ds.train, m, out, cl, cr, np.unique(np.rint(ds.train.rating).astype(np.int64)))
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("name,k", [("tiny", 7), ("ragged", 12)])
def test_objective_grad_hv_V(name, k, solver):
    ds = dataset(name)
    lam = 30.0
    U, V = np_init(ds.d1, ds.d2, k, seed=2, scale=0.5)
    e, _, _ = make_engine(ds, k, lam, solver=solver, U=U, V=V)
    O = ob.oracle(); X = to_csr(ds.train)
    m = O.comp_m(X, U, V)
    obj = e.initial_objective()
    oo = O.objective_new(X, m, U, V, lam) if solver == 2 else O.pcr_objective(X, m, U, V, lam)
    assert abs(obj - oo) / abs(oo) < 1e-12
    g = e.grad_V()
    go = O.obtain_g_new(X, U, V, m, lam) if solver == 2 else O.pcr_obtain_g(X, U, V, m, lam)
    assert rel(g, go) < VEC_TOL
    a = np.random.default_rng(5).standard_normal(V.shape)
    h = e.hv_V(a)
    ho = O.compute_Ha_new(X, a, m, U, lam) if solver == 2 else O.pcr_compute_Ha(X, a, m, U, lam)
    assert rel(h, ho) < VEC_TOL
    e.close()


@pytest.mark.parametrize("name,k", [("tiny", 7), ("ragged", 12)])
def test_grad_hv_U(name, k):
    ds = dataset(name)
    lam = 30.0
    U, V = np_init(ds.d1, ds.d2, k, seed=4, scale=0.5)
    e, _, _ = make_engine(ds, k, lam, U=U, V=V)
    O = ob.oracle(); X = to_csr(ds.train)
    m = O.comp_m(X, U, V)
    g, obj = e.grad_U()
    S = np.random.default_rng(6).standard_normal(U.shape)
    HS = e.hv_U(S)
    rp = ds.train.row_ptr
    for u in range(ds.d1):
        a, b = int(rp[u]), int(rp[u + 1])
        go, oo, ho = O.user_stage(X.rows[a:b], X.vals[a:b], m[a:b], V, lam, U[u], S[u])
        assert rel(g[u], go) < VEC_TOL if np.abs(go).max() > 0 else np.abs(g[u]).max() == 0, u
        assert abs(obj[u] - oo) <= 1e-12 * max(abs(oo), 1.0), u
        if b > a:
            assert rel(HS[u], ho) < VEC_TOL, u
    e.close()


@pytest.mark.parametrize("which", [0, 1])
@pytest.mark.parametrize("name", ["tiny", "ragged", "ragged_real"])
def test_eval(name, which):
    ds = dataset(name)
    k = 9
    U, V = np_init(ds.d1, ds.d2, k, seed=8, scale=0.7)
    e, _, _ = make_engine(ds, k, 10.0, U=U, V=V, levels=(name != "ragged_real"))
    R = ds.train if which == 0 else ds.test
    got = e.eval(which)
    want = ob.oracle().eval(to_csr(R), U, V, 10)
    assert abs(got[0] - want[0]) < 1e-12
    assert abs(got[1] - want[1]) < 1e-12
    e.close()


@pytest.mark.parametrize("name", ["tiny", "ragged", "ragged_real"])
def test_eval_pair_counts_sorted_vs_all_pairs(name):
    """The O(len * levels) pair-error count from the Primal-CR++ sorted state (SURVEY App. A) is the SAME integer, user by
    user, as the all-pairs kernel and as the reference's O(len^2) loop (util.cpp:467-479) -- with exact score ties
    (duplicated item rows, an all-zero user row: `>=` counts ties as errors) and a heavy user of 5000 ratings.  With
    real-valued ratings lround levels do not order the ratings, so the sorted path must refuse and the exact-double
    all-pairs count stays in charge."""
    ds = dataset(name)
    k = 5
    U, V = np_init(ds.d1, ds.d2, k, seed=13, scale=0.7)
    rp = ds.train.row_ptr
    big = int(np.argmax(np.diff(rp)))
    its = ds.train.item[rp[big]:rp[big + 1]]
    V[its[1::7]] = V[its[0]]                      # many exactly equal scores inside the heaviest user (and others)
    U[min(10, ds.d1 - 1)] = 0.0                   # a user whose scores all tie at 0
    e, _, _ = make_engine(ds, k, 10.0, U=U, V=V, levels=(name != "ragged_real"))
    want, counts, per_user = ob.oracle().eval(to_csr(ds.train), U, V, 10, want_counts=True)
    err0, ndcg0, c0 = e.eval_error_counts(0, method=0)
    assert np.array_equal(c0, per_user)
    assert abs(err0 - want[0]) < 1e-12 and abs(ndcg0 - want[1]) < 1e-12
    if name == "ragged_real":
        with pytest.raises(api.PrimalCRError, match="integer ratings"):
            e.eval_error_counts(0, method=1)
    else:
        err1, ndcg1, c1 = e.eval_error_counts(0, method=1)
        assert np.array_equal(c1, per_user)
        assert err1 == err0 and ndcg1 == ndcg0
        e.initial_objective()                      # sorted state now exists: plain eval() takes the sorted path by itself
        assert e.eval(0) == (err0, ndcg0)
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("name,k,lam", [("tiny", 7, 50.0), ("ragged", 10, 20.0), ("tiny", 100, 5000.0)])
def test_update_V_then_U(name, k, lam, solver):
    """One outer iteration, stage by stage: V, U, objectives and the integer control-flow counters."""
    ds = dataset(name)
    e, U, V = make_engine(ds, k, lam, solver=solver)
    O = ob.oracle(); X = to_csr(ds.train)
    res = O.train(solver, X, None, U, V, lam, 1, do_predict=0)
    oV = e.update_V()
    oU = e.update_U()
    c = e.counters()
    Ug, Vg = e.get_factors()
    cnt = res["counters"][0]
    assert (c["v_cg_iters"], c["v_ls_trials"], c["v_ls_accepted"]) == tuple(cnt[:3])
    assert (c["u_cg_len_sum"], c["u_ls_len_sum"], c["u_skipped"], c["u_cg_iters"], c["u_ls_trials"]) == tuple(cnt[3:8])
    assert abs(oU - res["obj"][1]) / abs(res["obj"][1]) < OBJ_TOL
    assert rel(Vg, res["V"]) < 1e-8
    assert rel(Ug, res["U"]) < 1e-8
    assert oV > 0
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("stepsize", [48.0, 1.0e6])
def test_line_search_branches(stepsize, solver):
    """The rarely taken control-flow branches (SURVEY 7, "control-flow parity"), forced through parameter.stepsize
    (pmf.h:9-49; not settable from the CLI): 48 -> both line searches halve 5-6 times before accepting (48 and not 64:
    a halving sequence that hits exactly twice the Newton step makes f(u - 2 delta) = f(u) up to rounding for users
    whose loss is locally quadratic, and the strict `<` of pcrpp.cpp:808 is then decided by rounding noise); 1e6 -> the first
    V line search rejects all 20 trials (V kept, the scores of the last trial stay in m, pcrpp.cpp:443) and every user
    runs 20 U trials and keeps the last one (:814).  Also covers the fall-back of the score / sort reuse in update_V."""
    ds = dataset("tiny")
    k, lam = 7, 50.0
    U, V = init_factors(ds.d1, ds.d2, k)
    res = ob.oracle().train(solver, to_csr(ds.train), None, U, V, lam, 3, do_predict=0, stepsize=stepsize)
    e = api.Engine(api.Parameter(solver_type=solver, k=k, lambda_=lam, maxiter=3, stepsize=stepsize))
    e.set_levels(np.unique(np.rint(ds.train.rating).astype(np.int64)))
    e.set_train(ds.train); e.set_factors(U, V)
    assert abs(e.initial_objective() - res["obj"][0]) <= OBJ_TOL * abs(res["obj"][0])
    seen_rejected = False
    for i in (1, 2, 3):
        o = e.outer_iteration()
        c = e.counters(); cnt = res["counters"][i - 1]
        assert (c["v_cg_iters"], c["v_ls_trials"], c["v_ls_accepted"]) == tuple(int(x) for x in cnt[:3]), (i, c, cnt)
        assert (c["u_cg_len_sum"], c["u_ls_len_sum"], c["u_skipped"], c["u_cg_iters"], c["u_ls_trials"]) == tuple(int(x) for x in cnt[3:8]), (i, c, cnt)
        assert abs(o - res["obj"][i]) <= 1e-8 * abs(res["obj"][i]), (i, o, res["obj"][i])
        seen_rejected |= c["v_ls_accepted"] == 0
    assert c["v_ls_trials"] > 1                       # the branch this test is about was really taken
    assert seen_rejected == (stepsize > 1e3)
    Ug, Vg = e.get_factors()
    assert rel(Ug, res["U"]) < 1e-7 and rel(Vg, res["V"]) < 1e-7
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("name,k,lam,iters", [("tiny", 7, 50.0, 4), ("ragged", 10, 20.0, 3), ("ml1m", 10, 5000.0, 2),
                                              ("ml1m", 100, 5000.0, 1)])
def test_training_trajectory(name, k, lam, iters, solver):
    """The pcrpp()/pcr() driver: objective per outer iteration, pairwise error and NDCG@10 vs the oracle."""
    ds = dataset(name)
    U, V = init_factors(ds.d1, ds.d2, k)
    O = ob.oracle()
    res = O.train(solver, to_csr(ds.train), to_csr(ds.test), U, V, lam, iters, do_predict=1)
    p = api.Parameter(solver_type=solver, k=k, lambda_=lam, maxiter=iters, do_predict=1)
    Ug, Vg = U.copy(), V.copy()
    lines = (api.pcrpp if solver == 2 else api.pcr)(ds.train, Ug, Vg, ds.test, p, log=None)
    objs = [float(l.split()[-1]) for l in lines if l.startswith("Iter ")]
    assert len(objs) == iters + 1
    for a, b in zip(objs, res["obj"]):
        assert abs(a - b) <= 1e-5 * abs(b)          # the log line carries 6 significant digits
    tr = [l for l in lines if l.startswith("(Training)")]
    te = [l for l in lines if l.startswith("(Testing)")]
    assert len(tr) == iters + 1 and len(te) == iters + 1
    for i in range(iters + 1):
        assert abs(float(tr[i].split()[4]) - res["evals"][i, 0]) < 1e-5
        assert abs(float(te[i].split()[-1]) - res["evals"][i, 3]) < NDCG_TOL
    assert rel(Ug, res["U"]) < 1e-7 and rel(Vg, res["V"]) < 1e-7
    # full-precision objective through the stage API
    e, _, _ = make_engine(ds, k, lam, solver=solver, U=U, V=V, maxiter=iters)
    assert abs(e.initial_objective() - res["obj"][0]) / res["obj"][0] < OBJ_TOL
    for i in range(1, iters + 1):
        o = e.outer_iteration()
        assert abs(o - res["obj"][i]) / res["obj"][i] < OBJ_TOL, i
        err, ndcg = e.eval(1)
        assert abs(ndcg - res["evals"][i, 3]) < NDCG_TOL
        assert abs(err - res["evals"][i, 2]) < 1e-9
    e.close()


def test_pcr_vs_pcrpp_self_consistency():
    """T3 of SURVEY section 4: on data where every user has two distinct ratings the two solvers minimise the same
    objective; their device objectives must agree to ~1e-12 at the same point."""
    ds = dataset("tiny")
    k, lam = 8, 40.0
    U, V = np_init(ds.d1, ds.d2, k, seed=21, scale=0.5)
    e2, _, _ = make_engine(ds, k, lam, solver=2, U=U, V=V)
    e1, _, _ = make_engine(ds, k, lam, solver=1, U=U, V=V)
    a, b = e2.initial_objective(), e1.initial_objective()
    assert abs(a - b) / abs(a) < 1e-12
    assert rel(e2.grad_V(), e1.grad_V()) < 1e-10
    e1.close(); e2.close()


def test_large_scale_properties():
    """Size-independent checks at a size the CPU oracle cannot reach quickly (ml1m-shape x k=100):
    the objective the solver reports after update_U equals the objective recomputed from scratch, decreases
    monotonically, and Primal-CR / Primal-CR++ agree on it."""
    ds = dataset("ml1m")
    k, lam = 100, 5000.0
    e, U, V = make_engine(ds, k, lam, solver=2)
    prev = e.initial_objective()
    for _ in range(2):
        now = e.outer_iteration()
        assert now < prev
        again = e.initial_objective()           # recompute scores + sort + sweep from the new U, V
        assert abs(again - now) / now < 1e-10
        prev = now
    Ug, Vg = e.get_factors()
    e1, _, _ = make_engine(ds, k, lam, solver=1, U=Ug, V=Vg)
    assert abs(e1.initial_objective() - prev) / prev < 1e-10
    e.close(); e1.close()


@pytest.mark.parametrize("solver", [2, 1])
@pytest.mark.parametrize("name", ["tiny", "ml1m600", "toy400"])
def test_golden_fixture_from_the_reference(name, solver):
    """CUDA path against outputs of the UNMODIFIED reference (tests/golden/*.npz): stage outputs at the initial
    point, objective / error / NDCG per outer iteration, final factors.  toy400 has real-valued ratings (9 lround
    levels for Primal-CR++, exact-double comparisons for Primal-CR and the evaluation)."""
    import os
    from primalcr_b200.data import Ratings
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_%s.npz" % name))
    d1, d2, k, lam, iters = int(g["d1"]), int(g["d2"]), int(g["k"]), float(g["lam"]), int(g["iters"])
    train = Ratings(d1, d2, g["row_ptr"], g["item"], g["rating"])
    p = api.Parameter(solver_type=solver, k=k, lambda_=lam, maxiter=iters)
    e = api.Engine(p)
    e.set_train(train)                      # level table derived by the library itself here
    has_test = len(g["t_item"]) > 0
    if has_test:
        e.set_test(Ratings(d1, d2, g["t_row_ptr"], g["t_item"], g["t_rating"]))
    e.set_factors(g["U0"], g["V0"])
    assert rel(e.scores(), g["m0"]) < 1e-13
    o0 = e.initial_objective()
    assert abs(o0 - float(g["obj%d" % solver])) <= 1e-12 * o0
    assert rel(e.grad_V(), g["g%d" % solver]) < VEC_TOL
    assert rel(e.hv_V(g["dir_a"]), g["Ha%d" % solver]) < VEC_TOL
    tr = e.eval(0)
    assert np.allclose(tr, g["eval_train0"], rtol=0, atol=1e-12)
    want, evals = g["s%d_obj" % solver], g["s%d_evals" % solver]
    # toy400: users whose ratings all round to ONE level (Primal-CR++) or whose few pairs are already separated by the
    # margin (both solvers) have a zero loss gradient, so the Newton step sends u_i to ~1e-17 (pure rounding noise, in
    # the reference too) and the ORDER of their scores -- hence their evaluation pairs -- is noise.  The all-users
    # numbers are therefore only compared loosely; the fixture's "test set" is the training set WITHOUT those 28 users
    # (make_golden.py), and that masked evaluation is held to the normal 1e-9 / 1e-4 below (has_test branch).
    err_tol, ndcg_tol = (0.03, 0.03) if name == "toy400" else (1e-9, NDCG_TOL)
    for i in range(1, iters + 1):
        o = e.outer_iteration()
        assert abs(o - want[i]) <= OBJ_TOL * abs(want[i]), i
        err, ndcg = e.eval(0)
        assert abs(err - evals[i, 0]) < err_tol and abs(ndcg - evals[i, 1]) < ndcg_tol
        if has_test:
            err, ndcg = e.eval(1)
            assert abs(err - evals[i, 2]) < 1e-9 and abs(ndcg - evals[i, 3]) < NDCG_TOL
    U, V = e.get_factors()
    assert rel(U, g["s%d_U" % solver]) < 1e-7 and rel(V, g["s%d_V" % solver]) < 1e-7
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
def test_dropin_cli_reference_main_with_our_solver(tmp_path, solver):
    """The reference's UNMODIFIED pmf-train.cpp linked against our pcr()/pcrpp() (shim + libprimalcr_b200.so):
    same command line, same data directory, same stdout lines (6 digits) and the same model file layout."""
    import os
    import subprocess
    from primalcr_b200.data import Dataset, Ratings, load_model, write_reference_dir
    exe = ob.ref_cli("gpu-omp-pmf-train")
    if exe is None:
        pytest.skip("oracle/_ref/gpu-omp-pmf-train was not built (needs /root/reference at build time)")
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "golden_tiny.npz"))
    d1, d2, k, lam, iters = int(g["d1"]), int(g["d2"]), int(g["k"]), float(g["lam"]), int(g["iters"])
    ds = Dataset(Ratings(d1, d2, g["row_ptr"], g["item"], g["rating"]), Ratings(d1, d2, g["t_row_ptr"], g["t_item"], g["t_rating"]))
    write_reference_dir(str(tmp_path / "data"), ds)
    out = subprocess.run([exe, "-s", str(solver), "-k", str(k), "-l", str(lam), "-t", str(iters), "-p", "1", "-n", "1",
                          str(tmp_path / "data"), str(tmp_path / "model")], cwd=tmp_path, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    ours = [l for l in out.stdout.splitlines() if l.startswith(("Iter", "(Training)", "(Testing)"))]
    ref = [l for l in str(g["s%d_stdout" % solver]).splitlines() if l.startswith(("Iter", "(Training)", "(Testing)"))]
    assert len(ours) == len(ref) == 3 * (iters + 1)
    # every other stdout line is byte-identical to the reference's (SURVEY App. B "exact strings"), "using 1 threads. " included
    fixed = lambda ls: [l for l in ls if not l.startswith(("Iter", "(Training)", "(Testing)", "Wall-time"))]
    assert fixed(out.stdout.splitlines()) == fixed(str(g["s%d_stdout" % solver]).splitlines())
    for a, b in zip(ours, ref):
        ta, tb = a.split(), b.split()
        assert ta[0] == tb[0]
        if ta[0] == "Iter":
            assert ta[1] == tb[1] and abs(float(ta[-1]) - float(tb[-1])) <= 2e-5 * abs(float(tb[-1]))
        else:
            assert abs(float(ta[4]) - float(tb[4])) < 2e-5 and abs(float(ta[-1]) - float(tb[-1])) < NDCG_TOL
    U, V = load_model(str(tmp_path / "model"))
    assert U.shape == (d1, k) and V.shape == (d2, k)
    assert rel(U, g["s%d_U" % solver]) < 1e-7 and rel(V, g["s%d_V" % solver]) < 1e-7
    assert os.path.exists(tmp_path / ("U.txt" if solver == 2 else "U%d.txt" % int(lam)))


@pytest.mark.parametrize("solver", [2, 1])
def test_own_cli_train_and_predict(tmp_path, solver):
    """primalcr-train / primalcr-predict (our C++ host CLI: fast loader + C ABI) against the reference CLI's golden
    stdout, model file, and the reference predictor's output format."""
    import os
    import subprocess
    from primalcr_b200.data import Dataset, Ratings, load_model, write_reference_dir
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "primalcr_b200", "bin", "primalcr-train")
    pexe = os.path.join(root, "primalcr_b200", "bin", "primalcr-predict")
    assert os.path.exists(exe) and os.path.exists(pexe), "run __graft_entry__.build()"
    g = np.load(os.path.join(root, "tests", "golden", "golden_tiny.npz"))
    d1, d2, k, lam, iters = int(g["d1"]), int(g["d2"]), int(g["k"]), float(g["lam"]), int(g["iters"])
    ds = Dataset(Ratings(d1, d2, g["row_ptr"], g["item"], g["rating"]), Ratings(d1, d2, g["t_row_ptr"], g["t_item"], g["t_rating"]))
    write_reference_dir(str(tmp_path / "data"), ds)
    out = subprocess.run([exe, "-s", str(solver), "-k", str(k), "-l", str(lam), "-t", str(iters), "-p", "1", "-n", "2",
                          str(tmp_path / "data"), str(tmp_path / "model")], cwd=tmp_path, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    ref_lines = str(g["s%d_stdout" % solver]).splitlines()
    ours = out.stdout.splitlines()
    assert ours[0] == ref_lines[0] and ours[1] == ref_lines[1] and ours[2] == ref_lines[2]     # rank / rows+cols / nnz header
    assert "using 2 threads. " in ours                  # pcrpp.cpp:855 verbatim (the reference run behind the fixture used -n 1)
    pick = lambda ls: [l for l in ls if l.startswith(("Iter", "(Training)", "(Testing)"))]
    for a, b in zip(pick(ours), pick(ref_lines)):
        ta, tb = a.split(), b.split()
        assert ta[0] == tb[0]
        if ta[0] == "Iter":
            assert abs(float(ta[-1]) - float(tb[-1])) <= 2e-5 * abs(float(tb[-1]))
        else:
            assert abs(float(ta[4]) - float(tb[4])) < 2e-5 and abs(float(ta[-1]) - float(tb[-1])) < NDCG_TOL
    assert len(pick(ours)) == len(pick(ref_lines))
    U, V = load_model(str(tmp_path / "model"))
    assert rel(U, g["s%d_U" % solver]) < 1e-7 and rel(V, g["s%d_V" % solver]) < 1e-7
    txt = np.loadtxt(tmp_path / ("U.txt" if solver == 2 else "U%d.txt" % int(lam)))
    assert txt.shape == (d1, k) and np.allclose(txt, U, rtol=2e-5, atol=1e-12)
    # predict: same "%lf" lines as omp-pmf-predict
    write = tmp_path / "data" / "test.ratings"
    r = subprocess.run([pexe, str(write), str(tmp_path / "model"), str(tmp_path / "pred")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    pred = np.loadtxt(tmp_path / "pred")
    T = ds.test
    want = np.einsum("ij,ij->i", U[T.users()], V[T.item])
    assert np.allclose(pred, want, atol=1e-6)
    assert np.allclose(api.predict(U, V, T.users(), T.item), want, rtol=1e-13, atol=1e-13)
    refp = ob.ref_cli("omp-pmf-predict")
    if refp:
        subprocess.run([refp, str(write), str(tmp_path / "model"), str(tmp_path / "pred_ref")], check=True)
        assert open(tmp_path / "pred").read() == open(tmp_path / "pred_ref").read()        # byte-identical output file
    # warm start (-w): one more iteration from the saved model continues the same trajectory
    out2 = subprocess.run([exe, "-s", str(solver), "-k", str(k), "-l", str(lam), "-t", "1", "-p", "0", "-w", str(tmp_path / "model"),
                           str(tmp_path / "data"), str(tmp_path / "model2")], cwd=tmp_path, capture_output=True, text=True)
    assert out2.returncode == 0, out2.stderr
    o = [float(l.split()[-1]) for l in out2.stdout.splitlines() if l.startswith("Iter ")]
    assert abs(o[0] - float(g["s%d_obj" % solver][iters])) <= 2e-5 * o[0] and o[1] < o[0]


def _custom_dataset(lens, d2, levels, seed):
    from primalcr_b200.data import Dataset, Ratings
    rng = np.random.default_rng(seed)
    users, items, vals = [], [], []
    for u, n in enumerate(lens):
        users.append(np.full(n, u)); items.append(np.sort(rng.choice(d2, size=n, replace=False)))
        vals.append(rng.integers(1, levels + 1, size=n).astype(np.float64))
    d1 = len(lens)
    tr = Ratings.from_coo(d1, d2, np.concatenate(users), np.concatenate(items), np.concatenate(vals)) if sum(lens) else Ratings.empty(d1, d2)
    return Dataset(tr, Ratings.empty(d1, d2))


@pytest.mark.parametrize("levels,k,heavy", [(7, 9, False), (2, 4, False), (8, 3, False), (12, 5, False),
                                            (8, 4, True), (5, 6, True), (3, 5, True), (11, 3, True),
                                            (40, 4, False), (101, 3, True), (256, 3, True)])
def test_level_count_variants(levels, k, heavy):
    """2, 7 and 8 rating levels go through the tile kernels (5- and 8-level instantiations, two- and three-word packed
    records), 12 / 40 / 101 (a 0-100 scale) / 256 levels through the per-user T-vector kernels (the reference's
    find_levels pcrpp.cpp:38-49 has no cap): two outer iterations against the oracle for each.  heavy: adds a
    2000-, a 4500- and a 9000-rating user (large tile / per-user class, and 3 / 5 chunks of the chunk-parallel path)."""
    lens = [0, 3, 40, 1, 700, 129, 1500, 64, 2, 31]
    d2 = 2000
    if heavy:
        lens = lens + [2000, 4500, 5, 9000, 17]
        d2 = 12000
    ds = _custom_dataset(lens, d2, levels, seed=levels)
    lam = 15.0
    e, U, V = make_engine(ds, k, lam, test=False)
    res = ob.oracle().train(2, to_csr(ds.train), None, U, V, lam, 2, do_predict=0)
    assert abs(e.initial_objective() - res["obj"][0]) <= OBJ_TOL * res["obj"][0]
    for i in (1, 2):
        o = e.outer_iteration()
        assert abs(o - res["obj"][i]) <= OBJ_TOL * res["obj"][i], (levels, i)
        c = e.counters(); cnt = res["counters"][i - 1]
        assert (c["v_cg_iters"], c["v_ls_trials"], c["u_cg_len_sum"], c["u_ls_len_sum"], c["u_skipped"]) == \
            (cnt[0], cnt[1], cnt[3], cnt[4], cnt[5])
    Ug, Vg = e.get_factors()
    assert rel(Ug, res["U"]) < 1e-7 and rel(Vg, res["V"]) < 1e-7
    e.close()


@pytest.mark.parametrize("solver", [2, 1])
def test_empty_and_degenerate_inputs(solver):
    """No ratings at all, a single rating, a single user: the reference's loops simply do not execute; U and V only
    feel the regulariser.  Must not crash, hang or produce NaN, and must agree with the oracle."""
    from primalcr_b200.data import Dataset, Ratings
    for lens in ([0, 0, 0], [0, 1, 0], [5]):
        ds = _custom_dataset(lens, 6, 3, seed=1)
        k, lam = 3, 2.0
        U, V = np_init(ds.d1, ds.d2, k, seed=1)
        e, _, _ = make_engine(ds, k, lam, solver=solver, U=U, V=V, test=False, levels=False)
        res = ob.oracle().train(solver, to_csr(ds.train) if ds.train.nnz else ob.Csr.empty(ds.d1, ds.d2), None, U, V, lam, 1, do_predict=0)
        o0 = e.initial_objective(); o1 = e.outer_iteration()
        assert np.isfinite(o0) and np.isfinite(o1)
        assert abs(o0 - res["obj"][0]) <= 1e-12 * max(res["obj"][0], 1.0)
        assert abs(o1 - res["obj"][1]) <= 1e-9 * max(res["obj"][1], 1.0)
        Ug, Vg = e.get_factors()
        assert np.abs(Ug - res["U"]).max() < 1e-9 and np.abs(Vg - res["V"]).max() < 1e-9
        e.close()


def test_bad_inputs_are_rejected():
    from primalcr_b200.data import Ratings
    p = api.Parameter(k=4)
    e = api.Engine(p)
    bad = Ratings(2, 5, np.array([0, 1, 2], np.int64), np.array([1, 7], np.int32), np.array([1.0, 2.0]))
    with pytest.raises(api.PrimalCRError, match="out of range"):
        e.set_train(bad)
    e.close()
    e = api.Engine(p)
    with pytest.raises(api.PrimalCRError):
        e.initial_objective()                 # nothing loaded yet
    many = Ratings(1, 400, np.array([0, 300], np.int64), np.arange(300, dtype=np.int32), np.arange(300, dtype=np.float64))
    with pytest.raises(api.PrimalCRError, match="256"):
        e.set_train(many)                     # more than 256 distinct lround levels: the 8-bit level index of Primal-CR++
    e.close()
    e = api.Engine(api.Parameter(k=4, solver_type=1))
    e.set_train(many)                         # Primal-CR compares exact ratings (pcr.cpp:23): no level table, no limit
    e.close()
    for bad_param in (dict(k=0), dict(k=257), dict(ndcg_k=65), dict(ndcg_k=0)):
        with pytest.raises(api.PrimalCRError):
            api.Engine(api.Parameter(**bad_param))
    # factor buffers reach the C ABI as raw pointers: wrong dtype / layout / shape must raise, not corrupt memory
    ds = dataset("tiny")
    e = api.Engine(api.Parameter(k=4))
    e.set_train(ds.train)
    U, V = np_init(ds.d1, ds.d2, 4)
    e.set_factors(U, V)
    for Ub, Vb in ((U.astype(np.float32), V), (np.asfortranarray(U), V), (U[:, :3], V), (U, V[::2]), (U[:-1], V)):
        with pytest.raises(api.PrimalCRError, match="C-contiguous float64"):
            e.get_factors(Ub, Vb)
    e.close()
    with pytest.raises(api.PrimalCRError, match="C-contiguous float64"):
        api.pcrpp(ds.train, U.astype(np.float32), V, None, api.Parameter(k=4), log=None)


@pytest.mark.parametrize("name,k", [("tiny", 7), ("ragged", 10)])
def test_l2_block_ordered_work_lists(name, k, monkeypatch):
    """With a (artificially tiny) L2 block size the CSC work units switch to their user-block-major order (the Yahoo /
    power-law shapes take this path at full size): results must not change."""
    monkeypatch.setenv("PRIMALCR_UBLOCK_MB", "0.002")
    ds = dataset(name)
    lam = 25.0
    e, U, V = make_engine(ds, k, lam, test=False)
    res = ob.oracle().train(2, to_csr(ds.train), None, U, V, lam, 2, do_predict=0)
    assert abs(e.initial_objective() - res["obj"][0]) <= OBJ_TOL * res["obj"][0]
    O = ob.oracle(); X = to_csr(ds.train)
    m = O.comp_m(X, U, V)
    assert rel(e.grad_V(), O.obtain_g_new(X, U, V, m, lam)) < VEC_TOL
    g, _ = e.grad_U()
    for u in range(0, ds.d1, max(1, ds.d1 // 10)):
        a, b = int(ds.train.row_ptr[u]), int(ds.train.row_ptr[u + 1])
        go, _, _ = O.user_stage(X.rows[a:b], X.vals[a:b], m[a:b], V, lam, U[u], U[u])
        assert rel(g[u], go) < VEC_TOL or np.abs(go).max() == 0
    for i in (1, 2):
        o = e.outer_iteration()
        assert abs(o - res["obj"][i]) <= OBJ_TOL * res["obj"][i]
    Ug, Vg = e.get_factors()
    assert rel(Ug, res["U"]) < 1e-7 and rel(Vg, res["V"]) < 1e-7
    e.close()
