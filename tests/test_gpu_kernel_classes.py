"""Every rank class and every sort path of the training kernels against the CPU oracle.

The training kernels are template instantiations chosen by the rank k (score gathers, row sums, the U-side CG vectors)
and by the length of a user and the number of rating levels T (tiles of three geometries, per-user sorts, heavy-user
chunk sort and merge).  The tests here reach every one of them and compare it with the oracle:

* rank sweep: k on both sides of every class boundary (kernel_classes() below states the dispatch table) on `ragged`
  plus 800 users of 48 popular items (more than 256 raters per item, so item columns split into several row-sum units);
* size classes: users of 0 ... 16385 ratings at T = 2, 5, 6, 8, 9, 12 with planted scores: integer ties (P1),
  float32-colliding runs that need the tile sort's exact fix-up or its fall-back network (P2), scores whose float32
  image is +-inf (P3).

Main tool: exact arithmetic.  With U, V, directions in {-1, 0, 1}, integer ratings, integer lambda and integer planted
scores every score, coefficient, objective, gradient and Hessian-vector product is an integer far below 2^53, hence
exact in any summation order, and the GPU must equal the oracle bit for bit.  test_*_are_exact_integers (no GPU) keeps
that premise true.  Real-valued runs of the same stages use the usual bars.
"""
import numpy as np
import pytest

from oracle import bindings as ob
from primalcr_b200 import api
from primalcr_b200.data import Dataset, Ratings, csr_in_file_order
from tests.test_gpu_parity import OBJ_TOL, VEC_TOL, check_sorted_state, make_engine
from tests.test_gpu_recommend import eligible, ref_topn
from tests.util import dataset, np_init, rel, to_csr

gpu = pytest.mark.gpu

LAM = 4.0                # integer lambda: lambda * V and the regulariser stay integers


# ----------------------------------------------------------------------------- the dispatch table
def kernel_classes(k):
    """Template instantiation every rank-dependent launcher picks for rank k (csrc/k_core.cu).

    nch = ceil(k / 2) 16-byte chunks of payload per factor row, ld = ceil16(k) the padded row length (engine.cu)."""
    nch = (k + 1) // 2
    ld = (k + 15) & ~15
    if nch <= 56:                                   # k_dots_units :194-195: G = 8, NC = ceil(nch / 8), at most 7
        du = (8, min((nch + 7) // 8, 7))
    elif nch <= 112:                                # :196-197: G = 16, NC = ceil(nch / 16) in 4..7
        du = (16, min((nch + 15) // 16, 7))
    else:                                           # :198-199
        du = (32, 4)
    return dict(dots_units=du,
                rowsum=(nch + 31) // 32,                             # k_rowsum :330, NCH = ceil(nch / 32)
                u_vec=1 if ld <= 64 else (2 if ld <= 128 else 4),    # u_finalize_cg :945-947, u_init_vec :1023-1025
                dots=4 if nch <= 4 else 8)                           # k_dots :117-121 (test-set scores, predict)


ALL_CLASSES = dict(dots_units={(8, nc) for nc in range(1, 8)} | {(16, nc) for nc in range(4, 8)} | {(32, 4)},
                   rowsum={1, 2, 3, 4}, u_vec={1, 2, 4}, dots={4, 8})

# both sides of every class boundary; odd k leave a zero padding column inside the last 16-byte chunk
K_LIST = [1, 2, 8, 9, 16, 17, 32, 33, 48, 49, 63, 64, 65, 80, 81, 96, 97, 112, 113, 127, 128, 129, 160, 161, 192, 193,
          224, 225, 255, 256]
PCR_K = [17, 64, 65, 128, 129, 256]        # Primal-CR training (its oracle is O(len^2) per user)
UBLOCK_K = [33, 129, 256]


def test_class_table_is_covered():
    for name, want in ALL_CLASSES.items():
        assert {kernel_classes(k)[name] for k in K_LIST} == want, name
        assert {kernel_classes(k)[name] for k in range(1, 257)} == want, name        # the table has no other class
    # every boundary is tested from both sides
    for k in range(1, 256):
        if kernel_classes(k) != kernel_classes(k + 1):
            assert k in K_LIST and k + 1 in K_LIST, k
    for k in UBLOCK_K + PCR_K:
        assert k in K_LIST


# ----------------------------------------------------------------------------- data sets
_cache = {}


def ragged_popular():
    """`ragged` plus 800 users with 1-40 ratings each over 48 popular items (about 340 raters per popular item, so its
    CSC column is cut into several row-sum units; `ragged` alone has at most 24 raters per item).  Five levels."""
    if "rp" not in _cache:
        base = dataset("ragged")
        d2 = base.d2
        rng = np.random.default_rng(41)
        pop = np.sort(rng.choice(d2, 48, replace=False))
        n_new = 800
        us, its, vs = [base.train.users()], [base.train.item], [base.train.rating]
        tu, ti, tv = [base.test.users()], [base.test.item], [base.test.rating]
        for q in range(n_new):
            u = base.d1 + q
            n = int(rng.integers(1, 41))
            us.append(np.full(n, u)); its.append(rng.choice(pop, n, replace=False))
            vs.append(rng.integers(1, 6, n).astype(np.float64))
            nt = int(rng.integers(0, 6))
            tu.append(np.full(nt, u)); ti.append(rng.choice(d2, nt, replace=False))
            tv.append(rng.integers(1, 6, nt).astype(np.float64))
        d1 = base.d1 + n_new
        train = Ratings.from_coo(d1, d2, np.concatenate(us), np.concatenate(its), np.concatenate(vs))
        test = csr_in_file_order(d1, d2, np.concatenate(tu), np.concatenate(ti), np.concatenate(tv))
        _cache["rp"] = Dataset(train, test, name="ragged_popular")
    return _cache["rp"]


# users of every size class, interleaved so that tiles open and close between classes; 16385 ratings = 9 heavy chunks
SIZE_LENS = [255, 2049, 1, 1024, 4097, 2, 256, 16385, 0, 1023, 6144, 2047, 257, 8193, 1025, 4095, 2048, 6145, 4096, 8192]
SIZE_D2 = 20000
T_LIST = [2, 5, 6, 8, 9, 12]


def size_dataset(T):
    """SIZE_LENS, then 130 consecutive short users (more than TILE_MAX_USERS = 128 in a row), then 800 users over 48
    popular items; integer ratings 1..T.  Items are the same for every T."""
    if ("size", T) not in _cache:
        rng = np.random.default_rng(7)
        lens = SIZE_LENS + list(rng.integers(1, 9, 130)) + list(rng.integers(1, 41, 800))
        pop = np.sort(rng.choice(SIZE_D2, 48, replace=False))
        us, its = [], []
        for u, n in enumerate(lens):
            us.append(np.full(n, u))
            its.append(rng.choice(pop, n, replace=False) if u >= len(SIZE_LENS) + 130 else rng.choice(SIZE_D2, n, replace=False))
        users, items = np.concatenate(us), np.concatenate(its)
        vals = np.random.default_rng(100 + T).integers(1, T + 1, len(users)).astype(np.float64)
        d1 = len(lens)
        _cache[("size", T)] = Dataset(Ratings.from_coo(d1, SIZE_D2, users, items, vals), Ratings.empty(d1, SIZE_D2),
                                      name="sizes_T%d" % T)
    return _cache[("size", T)]


def _user_of_len(n):
    return SIZE_LENS.index(n)


def int_inputs(d1, d2, k, seed):
    """U, V, a (V-side direction), S (U-side direction) with entries in {-1, 0, 1}."""
    rng = np.random.default_rng(seed)
    t = lambda r: rng.integers(-1, 2, size=(r, k)).astype(np.float64)
    return t(d1), t(d2), t(d2), t(d1)


# ----------------------------------------------------------------------------- planted scores (section sizes)
def plant_p1(R, seed):
    """Integer scores in [-3, 3]: ties everywhere, exact +-1 windows, ties across every heavy chunk boundary; -0.0 next
    to +0.0; every score of the 8193-rating user equal."""
    rng = np.random.default_rng(seed)
    m = rng.integers(-3, 4, R.nnz).astype(np.float64)
    z = np.flatnonzero(m == 0.0)
    m[z[::2]] = -0.0
    u = _user_of_len(8193)
    m[R.row_ptr[u]:R.row_ptr[u + 1]] = 2.0
    return m


# (user length, run length L, offset of the run inside the user): L = 40 is repaired by the tile sort's odd-even fix-up
# (L / 2 = 20 rounds), L = 300 needs 150 > 48 rounds, so that tile falls back to the exact network
P2_RUNS = [(1023, 40, 100), (1024, 300, 300), (2047, 40, 1000), (2048, 300, 1500), (4095, 40, 2000), (4096, 300, 10),
           (8193, 40, 2048 - 20), (16385, 300, 4 * 2048 - 150), (6144, 300, 6144 - 300)]


def plant_p2(R, seed):
    """Runs whose float32 images are all equal (0.75 + (L - j) 2^-45, j = 0..L-1: reversed index order, distinct
    doubles) inside users of each tile geometry and of the heavy path, with exact fp64 duplicates and +-0.0 in the same
    users; ordinary scores elsewhere."""
    rng = np.random.default_rng(seed)
    m = rng.standard_normal(R.nnz) * 2.0
    for n, L, off in P2_RUNS:
        a = int(R.row_ptr[_user_of_len(n)])
        j = np.arange(L)
        m[a + off:a + off + L] = 0.75 + (L - j) * 2.0 ** -45
        rest = np.setdiff1d(np.arange(a, a + n), np.arange(a + off, a + off + L))
        pick = rng.choice(rest, 12, replace=False)
        m[pick[:4]] = 0.75 + 7 * 2.0 ** -45          # exact duplicates of a run member
        m[pick[4:6]] = 0.75                            # the run's float image itself, as a double
        m[pick[6:9]] = 0.0
        m[pick[9:12]] = -0.0
    return m


def plant_p3(R, seed):
    """Scores beyond the float range (float32 image +-inf) next to ordinary ones, and the largest finite float."""
    rng = np.random.default_rng(seed)
    m = rng.standard_normal(R.nnz) * 2.0
    r = rng.random(R.nnz)
    m[r < 0.04] = 1e39
    m[(r >= 0.04) & (r < 0.08)] = -1e39
    m[(r >= 0.08) & (r < 0.10)] = 3.4e38
    m[(r >= 0.10) & (r < 0.11)] = 2e39
    return m


def test_planted_scores_premise():
    """What P2 relies on: a run's float32 images are equal, its doubles distinct, and the oracle sorts it reversed."""
    R = size_dataset(5).train
    m = plant_p2(R, 3)
    for n, L, off in P2_RUNS:
        a = int(R.row_ptr[_user_of_len(n)]) + off
        run = m[a:a + L]
        assert np.all(run.astype(np.float32) == np.float32(0.75)) and len(np.unique(run)) == L
        _, perm = ob.oracle().sorted_mm(run)
        assert np.array_equal(perm, np.arange(L)[::-1])
    m = plant_p3(R, 3)
    with np.errstate(over="ignore"):
        assert np.all(np.isinf(m[np.abs(m) > 3.5e38].astype(np.float32)))


# ----------------------------------------------------------------------------- oracle of the exact stages
def oracle_stages(R, U, V, a, S, m, lam, pcr=True):
    """Every stage output the exact checks compare, from the CPU oracle."""
    O = ob.oracle()
    X = to_csr(R)
    out = dict(obj=O.objective_new(X, m, U, V, lam), g=O.obtain_g_new(X, U, V, m, lam), Ha=O.compute_Ha_new(X, a, m, U, lam))
    gu = np.zeros_like(U); ou = np.zeros(R.d1); hu = np.zeros_like(U)
    rp = R.row_ptr
    for u in range(R.d1):
        b0, b1 = int(rp[u]), int(rp[u + 1])
        gu[u], ou[u], hu[u] = O.user_stage(X.rows[b0:b1], X.vals[b0:b1], m[b0:b1], V, lam, U[u], S[u])
    out.update(gu=gu, ou=ou, hu=hu)
    if pcr:
        out.update(pcr_obj=O.pcr_objective(X, m, U, V, lam), pcr_g=O.pcr_obtain_g(X, U, V, m, lam),
                   pcr_Ha=O.pcr_compute_Ha(X, a, m, U, lam))
    return out


def assert_exact_integers(out):
    for name, v in out.items():
        v = np.asarray(v, np.float64)
        assert np.all(np.isfinite(v)) and np.array_equal(v, np.rint(v)), name
        # 2^13 of headroom under 2^53 for partial sums that are larger than the result
        assert np.abs(v).max(initial=0.0) < 2.0 ** 40, (name, np.abs(v).max())


def rank_inputs(k):
    ds = ragged_popular()
    return ds, int_inputs(ds.d1, ds.d2, k, seed=1000 + k)


@pytest.mark.parametrize("k", K_LIST)
def test_rank_inputs_are_exact_integers(k):
    ds, (U, V, a, S) = rank_inputs(k)
    m = ob.oracle().comp_m(to_csr(ds.train), U, V)
    out = oracle_stages(ds.train, U, V, a, S, m, LAM)
    out["m"] = m
    assert_exact_integers(out)
    assert out["obj"] == out["pcr_obj"]            # integer ratings: both solvers minimise the same objective


@pytest.mark.parametrize("T", T_LIST)
def test_size_inputs_are_exact_integers(T):
    ds = size_dataset(T)
    U, V, a, S = int_inputs(ds.d1, ds.d2, 5, seed=T)
    out = oracle_stages(ds.train, U, V, a, S, plant_p1(ds.train, T), LAM, pcr=(T == 5))
    assert_exact_integers(out)


# ----------------------------------------------------------------------------- GPU: rank sweep
def check_exact_stages(ds, k, U, V, a, S, want):
    """Primal-CR++ and Primal-CR stage outputs at integer inputs: equal to the oracle's, not merely close."""
    X = to_csr(ds.train)
    e, _, _ = make_engine(ds, k, LAM, solver=2, U=U, V=V)
    m = e.scores()
    assert np.array_equal(m, ob.oracle().comp_m(X, U, V))
    assert e.initial_objective() == want["obj"]
    assert np.array_equal(e.grad_V(), want["g"])
    assert np.array_equal(e.hv_V(a), want["Ha"])
    g, obj = e.grad_U()
    assert np.array_equal(g, want["gu"])
    assert np.array_equal(obj, want["ou"])
    HS = e.hv_U(S)
    has = np.diff(ds.train.row_ptr) > 0                # users without ratings: Hs is not defined by the reference
    assert np.array_equal(HS[has], want["hu"][has])
    e.close()
    e, _, _ = make_engine(ds, k, LAM, solver=1, U=U, V=V, test=False)
    assert e.initial_objective() == want["pcr_obj"]
    assert np.array_equal(e.grad_V(), want["pcr_g"])
    assert np.array_equal(e.hv_V(a), want["pcr_Ha"])
    e.close()


@gpu
@pytest.mark.parametrize("k", K_LIST)
def test_rank_exact_stages(k):
    """Scores, objective, gradients and Hessian-vector products on both sides, test-set error counts, predict and
    recommend at every rank class, bit for bit."""
    ds, (U, V, a, S) = rank_inputs(k)
    O = ob.oracle()
    m = O.comp_m(to_csr(ds.train), U, V)
    check_exact_stages(ds, k, U, V, a, S, oracle_stages(ds.train, U, V, a, S, m, LAM))
    # pair-error counts: test set (scores by dots_kernel), training set (all pairs and from the sorted state)
    e, _, _ = make_engine(ds, k, LAM, solver=2, U=U, V=V)
    for which, R in ((1, ds.test), (0, ds.train)):
        want, _, per_user = O.eval(to_csr(R), U, V, 10, want_counts=True)
        err, _, c = e.eval_error_counts(which, method=0)
        assert np.array_equal(c, per_user), which
        assert abs(err - want[0]) < 1e-12, which
    _, _, c = e.eval_error_counts(0, method=1)
    assert np.array_equal(c, O.eval(to_csr(ds.train), U, V, 10, want_counts=True)[2])
    e.close()
    rng = np.random.default_rng(k)
    pu = rng.integers(0, ds.d1, 4000); pi = rng.integers(0, ds.d2, 4000)
    assert np.array_equal(api.predict(U, V, pu, pi), np.einsum("ij,ij->i", U[pu], V[pi]))
    users = np.concatenate([np.arange(24), rng.choice(np.arange(24, ds.d1), 176, replace=False)]).astype(np.int32)
    ok = eligible(ds.train, users, ds.d2)
    S_full = U[users] @ V.T
    for n in (10, 200):                                # 200: the topn kernel's other k-chunk width
        it, sc = api.recommend(U, V, n, exclude=ds.train, users=users)
        ri, rs = ref_topn(S_full, ok, n, exact=True)
        assert np.array_equal(it, ri), n
        assert np.array_equal(sc, rs, equal_nan=True), n


@gpu
@pytest.mark.parametrize("k", K_LIST)
def test_rank_real_valued_stages(k):
    """The same stages from real-valued factors and directions: nothing above depends on integer inputs."""
    ds = ragged_popular()
    U, V = np_init(ds.d1, ds.d2, k, seed=k, scale=(4.0 / k) ** 0.25)
    rng = np.random.default_rng(k + 1)
    a = rng.standard_normal(V.shape); S = rng.standard_normal(U.shape)
    lam = 7.3
    O = ob.oracle(); X = to_csr(ds.train)
    mo = O.comp_m(X, U, V)
    want = oracle_stages(ds.train, U, V, a, S, mo, lam, pcr=k in PCR_K)
    e, _, _ = make_engine(ds, k, lam, solver=2, U=U, V=V)
    assert rel(e.scores(), mo) < 1e-13
    assert abs(e.initial_objective() - want["obj"]) <= 1e-12 * abs(want["obj"])
    assert rel(e.grad_V(), want["g"]) < VEC_TOL
    assert rel(e.hv_V(a), want["Ha"]) < VEC_TOL
    g, obj = e.grad_U()
    HS = e.hv_U(S)
    for u in range(ds.d1):
        if ds.train.row_ptr[u + 1] > ds.train.row_ptr[u]:
            assert rel(g[u], want["gu"][u]) < VEC_TOL, u
            assert abs(obj[u] - want["ou"][u]) <= 1e-12 * max(abs(want["ou"][u]), 1.0), u
            assert rel(HS[u], want["hu"][u]) < VEC_TOL, u
    e.close()
    if k in PCR_K:
        e, _, _ = make_engine(ds, k, lam, solver=1, U=U, V=V, test=False)
        assert abs(e.initial_objective() - want["pcr_obj"]) <= 1e-12 * abs(want["pcr_obj"])
        assert rel(e.grad_V(), want["pcr_g"]) < VEC_TOL
        assert rel(e.hv_V(a), want["pcr_Ha"]) < VEC_TOL
        e.close()


def check_one_iteration(ds, k, solver):
    """update_V + update_U from real-valued factors against the oracle's first outer iteration: objective, the eight
    control-flow counters, factors."""
    lam = 20.0
    U, V = np_init(ds.d1, ds.d2, k, seed=3 * k, scale=(4.0 / k) ** 0.25)
    res = ob.oracle().train(solver, to_csr(ds.train), None, U, V, lam, 1, do_predict=0)
    e, _, _ = make_engine(ds, k, lam, solver=solver, U=U, V=V, test=False)
    e.update_V()
    oU = e.update_U()
    c = e.counters()
    cnt = res["counters"][0]
    assert (c["v_cg_iters"], c["v_ls_trials"], c["v_ls_accepted"]) == tuple(cnt[:3])
    assert (c["u_cg_len_sum"], c["u_ls_len_sum"], c["u_skipped"], c["u_cg_iters"], c["u_ls_trials"]) == tuple(cnt[3:8])
    assert abs(oU - res["obj"][1]) / abs(res["obj"][1]) < OBJ_TOL
    Ug, Vg = e.get_factors()
    assert rel(Vg, res["V"]) < 1e-8 and rel(Ug, res["U"]) < 1e-8
    e.close()


@gpu
@pytest.mark.parametrize("k", K_LIST)
def test_rank_one_iteration(k):
    check_one_iteration(ragged_popular(), k, 2)


@gpu
@pytest.mark.parametrize("k", PCR_K)
def test_rank_one_iteration_pcr(k):
    check_one_iteration(ragged_popular(), k, 1)


@gpu
@pytest.mark.parametrize("k", UBLOCK_K)
def test_user_block_major_units(k, monkeypatch):
    """The CSC row-sum units in their user-block-major order (a tiny L2 block): still bit for bit."""
    monkeypatch.setenv("PRIMALCR_UBLOCK_MB", "0.002")
    ds, (U, V, a, S) = rank_inputs(k)
    m = ob.oracle().comp_m(to_csr(ds.train), U, V)
    check_exact_stages(ds, k, U, V, a, S, oracle_stages(ds.train, U, V, a, S, m, LAM))


# ----------------------------------------------------------------------------- GPU: size classes and sort paths
def expected_route(T):
    """Kernels the sorted state of size_dataset(T) must launch (engine.cu set_train: tiles for T <= 8, the medium and
    large tile geometries only for T <= 5, per-user S / L / H kernels for T >= 9)."""
    present, absent = {"heavy_chunk_sort", "heavy_merge"}, set()
    if T <= 5:
        present |= {"tile_prepare", "tile_prepare_M", "tile_prepare_L", "hv_level_hist"}
        absent |= {"sort_users_S", "sort_users_L", "windows_S", "windows_L", "windows_H"}
    elif T <= 8:
        present |= {"tile_prepare", "sort_users_L", "windows_L", "hv_level_hist"}
        absent |= {"tile_prepare_M", "tile_prepare_L", "sort_users_S", "windows_S", "windows_H"}
    else:
        present |= {"sort_users_S", "sort_users_L", "windows_S", "windows_L", "windows_H"}
        absent |= {"tile_prepare", "tile_prepare_M", "tile_prepare_L", "hv_level_hist"}
    return present, absent


@gpu
@pytest.mark.parametrize("T", T_LIST)
def test_size_classes_sorted_state_and_stages(T):
    ds = size_dataset(T)
    R = ds.train
    k = 5
    U, V, a, S = int_inputs(ds.d1, ds.d2, k, seed=T)
    levels = np.arange(1, T + 1)
    e, _, _ = make_engine(ds, k, LAM, U=U, V=V, test=False)
    assert e.num_levels() == T
    e.profile_enable(True)
    has = np.diff(R.row_ptr) > 0
    for name, plant in (("P1", plant_p1), ("P2", plant_p2), ("P3", plant_p3)):
        m = plant(R, T)
        e.set_scores(m)
        e.profile_reset()
        g = e.grad_V()                                  # one sort of every user, then the sweeps
        prof = {n: v["launches"] for n, v in e.profile().items() if v["launches"] > 0}
        present, absent = expected_route(T)
        assert present <= set(prof), (name, present - set(prof))
        assert not (absent & set(prof)), (name, absent & set(prof))
        assert prof["heavy_merge"] == 4 * prof["heavy_chunk_sort"], prof        # 16385 ratings: 9 chunks, 4 passes
        out = e.sort_segments()
        cl, cr = e.level_counts()
        check_sorted_state(R, m, out, cl, cr, levels)
        if name == "P3":
            continue
        want = oracle_stages(R, U, V, a, S, m, LAM, pcr=False)
        obj = e.objective()
        Ha = e.hv_V(a)
        gu, ou = e.grad_U()
        hu = e.hv_U(S)
        if name == "P1":
            assert obj == want["obj"]
            assert np.array_equal(g, want["g"]) and np.array_equal(Ha, want["Ha"])
            assert np.array_equal(gu, want["gu"]) and np.array_equal(ou, want["ou"])
            assert np.array_equal(hu[has], want["hu"][has])
        else:
            assert abs(obj - want["obj"]) <= OBJ_TOL * abs(want["obj"])
            assert rel(g, want["g"]) < VEC_TOL and rel(Ha, want["Ha"]) < VEC_TOL
            assert rel(gu, want["gu"]) < VEC_TOL and rel(hu[has], want["hu"][has]) < VEC_TOL
            assert np.all(np.abs(ou - want["ou"]) <= 1e-12 * np.maximum(np.abs(want["ou"]), 1.0))
    e.close()


@gpu
def test_size_classes_pcr_stages():
    """Primal-CR objective, gradient and Hv of V on the size-class set with the P1 scores, bit for bit."""
    T, k = 5, 5
    ds = size_dataset(T)
    U, V, a, S = int_inputs(ds.d1, ds.d2, k, seed=T)
    m = plant_p1(ds.train, T)
    want = oracle_stages(ds.train, U, V, a, S, m, LAM, pcr=True)
    e, _, _ = make_engine(ds, k, LAM, solver=1, U=U, V=V, test=False)
    e.set_scores(m)
    assert e.objective() == want["pcr_obj"]
    assert np.array_equal(e.grad_V(), want["pcr_g"])
    assert np.array_equal(e.hv_V(a), want["pcr_Ha"])
    e.close()
