"""Similar items / users (primalcr_similar / api.similar / primalcr-similar) against a numpy reference.

With integer factors every dot product and squared norm is an exact integer, so sqrt, the one product of norms and the
one division are correctly rounded alike in numpy and CUDA: whole rows, ids and score bits, must equal the reference's
order (score descending, NaN last, ties to the smaller id).  Real-valued factors are judged by test_gpu_recommend's
tolerance and near-tie rules, and the dot measure against primalcr_recommend itself."""
import os
import subprocess

import numpy as np
import pytest

from primalcr_b200 import api
from primalcr_b200.data import Ratings, save_model
from tests.test_gpu_recommend import check_rows, eligible, random_exclusion

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIM = os.path.join(ROOT, "primalcr_b200", "bin", "primalcr-similar")
QNAN = np.array([0x7ff8000000000000], np.int64).view(np.float64)[0]


# ----------------------------------------------------------------------------- reference
def ref_scores(M, queries, measure):
    S = M[queries] @ M.T
    if measure == "cosine":
        nrm = np.sqrt(np.einsum("ij,ij->i", M, M))
        with np.errstate(divide="ignore", invalid="ignore"):
            S = S / (nrm[queries][:, None] * nrm[None, :])
    return S


def candidates(excl, queries, n):
    ok = eligible(excl, queries, n)
    ok[np.arange(len(queries)), queries] = False
    return ok


def ref_order(S, ok):
    """Every row of S in the library's total order, eligible entries first -> (ids, scores, eligible count)."""
    isn = np.isnan(S)
    neg = np.where(isn, 0.0, -S)
    ids = np.broadcast_to(np.arange(S.shape[1]), S.shape)
    order = np.lexsort((ids, neg, isn, ~ok), axis=-1)
    sc = np.take_along_axis(S, order, 1)
    sc = np.where(sc == 0.0, 0.0, sc)                   # returned as +0.0
    sc = np.where(np.isnan(sc), QNAN, sc)               # and one NaN
    return order.astype(np.int32), sc, ok.sum(1)


def ref_rows(order, sc, cnt, n):
    m = min(n, order.shape[1])
    ids = np.full((len(order), n), -1, np.int32); scores = np.full((len(order), n), QNAN)
    have = np.arange(m)[None, :] < cnt[:, None]
    ids[:, :m] = np.where(have, order[:, :m], -1)
    scores[:, :m] = np.where(have, sc[:, :m], QNAN)
    return ids, scores


def bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def similar_checked(M, n, measure, excl=None, queries=None):
    ids, sc = api.similar(M, n, measure=measure, exclude=excl, queries=queries)
    nq = M.shape[0] if queries is None else len(queries)
    assert ids.shape == (nq, n) and sc.shape == (nq, n) and ids.dtype == np.int32 and sc.dtype == np.float64
    return ids, sc


def assert_exact(M, measure, topns, excl=None, queries=None):
    q = np.arange(M.shape[0]) if queries is None else np.asarray(queries)
    order, sc, cnt = ref_order(ref_scores(M, q, measure), candidates(excl, q, M.shape[0]))
    for n in topns:
        ids, scores = similar_checked(M, n, measure, excl, queries)
        ri, rs = ref_rows(order, sc, cnt, n)
        assert np.array_equal(ids, ri), (measure, n)
        assert np.array_equal(bits(scores), bits(rs)), (measure, n)


def integer_factors(n, k, seed):
    """[-3, 3] integers with long exact tie runs, zero rows (+0.0 and -0.0 entries) and a negated row."""
    rng = np.random.default_rng(seed)
    M = rng.integers(-3, 4, size=(n, k)).astype(np.float64)
    if n >= 40:
        M[10:40] = M[9]                                  # 31 identical rows
        M[[3, 41 % n]] = 0.0
        M[n - 1] = -0.0
        M[5] = -M[4]
        M[7] = 2.0 * M[6]                                # cosine exactly 1 or the rounding of it
    return M


# ----------------------------------------------------------------------------- CPU
def test_similar_without_gpu_fails_loudly(have_gpu):
    if have_gpu:
        pytest.skip("a GPU is present")
    M = np.ones((5, 2))
    with pytest.raises(api.PrimalCRError, match="no CPU fallback|CUDA"):
        api.similar(M, 2)
    ids = np.empty((5, 2), np.int32)
    assert api.lib().primalcr_similar(M.ctypes.data, 5, 2, 1, None, None, None, 5, 2, ids.ctypes.data, None, 0) == -2


def test_unknown_measure_is_rejected_first():
    M = np.ones((5, 2))
    ids = np.empty((5, 2), np.int32)
    for m in (2, -1):
        assert api.lib().primalcr_similar(M.ctypes.data, 5, 2, m, None, None, None, 5, 2, ids.ctypes.data, None, 0) == -1
    with pytest.raises(api.PrimalCRError, match="measure"):
        api.similar(M, 2, measure="euclidean")


# ----------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu
TOPNS = (1, 32, 33, 128, 129, 256)


@gpu
@pytest.mark.parametrize("measure", ["cosine", "dot"])
@pytest.mark.parametrize("k", [1, 7, 8, 100, 255, 256])
def test_exact_integer_factors(measure, k):
    M = integer_factors(1300, k, seed=k)              # 1300 = 5 tiles of 256 + 20, 2 tiles of 512 + 276
    assert_exact(M, measure, TOPNS)


@gpu
@pytest.mark.parametrize("measure", ["cosine", "dot"])
def test_exact_small_and_ragged_n(measure):
    for n in (1, 2, 3, 63, 64, 65, 255, 257, 513):
        M = integer_factors(n, 8, seed=n)
        assert_exact(M, measure, (1, 33, 256))
    # the 1-row matrix: the query is its only row, so its row is all padding
    ids, sc = similar_checked(np.ones((1, 4)), 5, measure)
    assert np.all(ids == -1) and np.all(np.isnan(sc))


@gpu
def test_exact_with_exclusion_and_queries():
    rng = np.random.default_rng(4)
    n = 900
    M = integer_factors(n, 16, seed=99)
    excl = random_exclusion(n, n, rng, 500)
    q = rng.choice(n, size=300, replace=True).astype(np.int32)
    for measure in ("cosine", "dot"):
        assert_exact(M, measure, (5, 100, 256), excl=excl)
        assert_exact(M, measure, (5, 100, 256), excl=excl, queries=q)


@gpu
def test_zero_rows_give_nan_cosine_ordered_by_id():
    M = integer_factors(200, 12, seed=5)                # 199 candidates: the whole order fits in topn = 256
    M[[20, 100, 150]] = 0.0
    ids, sc = similar_checked(M, 256, "cosine")
    zero = [3, 20, 41, 100, 150, 199]
    for z in zero:                                     # a zero query: every score NaN, ids ascending without itself
        assert np.array_equal(ids[z, :199], [i for i in range(200) if i != z]) and np.all(np.isnan(sc[z]))
        assert np.all(ids[z, 199:] == -1)
    other = 0
    row_i, row_s = ids[other, :199], sc[other, :199]
    assert list(row_i[193:]) == zero and not np.any(np.isnan(row_s[:193]))   # zero rows rank last, by id
    assert np.array_equal(bits(sc[other, 193:]), bits(np.full(63, QNAN)))    # one NaN, padding included


@gpu
@pytest.mark.parametrize("scale", [1.0, 0.03, 40.0])
@pytest.mark.parametrize("measure", ["cosine", "dot"])
def test_real_valued_factors(measure, scale):
    rng = np.random.default_rng(int(scale * 100))
    n, k = 3000, 100
    M = rng.standard_normal((n, k)) * scale
    M[::7] *= 3.0                                      # uneven norms, as trained factors have
    excl = random_exclusion(n, n, rng, 30)
    q = np.arange(n)
    B = M / np.linalg.norm(M, axis=1)[:, None] if measure == "cosine" else M
    ok = candidates(excl, q, n)
    for topn in (10, 100, 256):
        ids, sc = similar_checked(M, topn, measure, excl)
        check_rows(ids, sc, B, B, ok, topn)


@gpu
def test_dot_equals_recommend_with_self_excluded():
    rng = np.random.default_rng(8)
    n, k = 2500, 32
    M = rng.standard_normal((n, k))
    M[[5, 6]] = M[4]; M[9] = 0.0; M[11] = np.nan
    excl = random_exclusion(n, n, rng, 40)
    us = np.concatenate([excl.users(), np.arange(n)])
    its = np.concatenate([excl.item.astype(np.int64), np.arange(n)])
    merged = Ratings.from_coo(n, n, us, its, np.ones(len(us)))
    for topn in (1, 32, 100, 200):
        ids, sc = similar_checked(M, topn, "dot", excl)
        ri, rs = api.recommend(M, M, topn, exclude=merged)
        assert np.array_equal(ids, ri) and np.array_equal(bits(sc), bits(rs)), topn


@gpu
def test_contract_edges():
    rng = np.random.default_rng(12)
    n, k = 700, 10
    M = rng.standard_normal((n, k))
    # q in its own exclusion row (repeated), and row 1 excluding every other row: an all-padding row
    us = [np.zeros(3, int), np.ones(n, int), np.full(4, 2)]
    its = [np.array([0, 0, 5]), np.arange(n), np.array([2, 2, 9, 9])]
    ex = Ratings.from_coo(n, n, np.concatenate(us), np.concatenate(its), np.ones(sum(len(x) for x in us)))
    for measure in ("cosine", "dot"):
        ids, sc = similar_checked(M, 256, measure, ex)
        assert not np.any(ids == np.arange(n)[:, None])
        assert not np.any(ids[0] == 5) and not np.any(np.isin(ids[2], [9])) and np.all(ids[[0, 2]] >= 0)
        assert np.all(ids[1] == -1) and np.all(np.isnan(sc[1]))
        B = M / np.linalg.norm(M, axis=1)[:, None] if measure == "cosine" else M
        check_rows(ids, sc, B, B, candidates(ex, np.arange(n), n), 256)
        # repeated and unordered queries: the rows of single-query calls, bit for bit
        q = np.array([699, 3, 3, 0, 1, 350, 699, 2], np.int32)
        sub_i, sub_s = similar_checked(M, 256, measure, ex, queries=q)
        assert np.array_equal(sub_i, ids[q]) and np.array_equal(bits(sub_s), bits(sc[q]))
        for j, u in enumerate(q[:4]):
            one_i, one_s = similar_checked(M, 256, measure, ex, queries=[u])
            assert np.array_equal(one_i[0], sub_i[j]) and np.array_equal(bits(one_s[0]), bits(sub_s[j]))
        # n_queries = 0
        z_i, z_s = similar_checked(M, 7, measure, ex, queries=np.zeros(0, np.int32))
        assert z_i.shape == (0, 7)
        # the same call twice
        again_i, again_s = similar_checked(M, 256, measure, ex)
        assert np.array_equal(again_i, ids) and np.array_equal(bits(again_s), bits(sc))


@gpu
def test_user_sized_matrix():
    """n = 300,000 rows of k = 100 (240 MB, more than L2): a query sample against every row."""
    rng = np.random.default_rng(31)
    n, k, topn = 300_000, 100, 50
    M = rng.standard_normal((n, k)) * 0.2
    q = np.sort(rng.choice(n, size=160, replace=False)).astype(np.int32)
    q = np.concatenate([q, [n - 1, 0]]).astype(np.int32)
    for measure in ("cosine", "dot"):
        ids, sc = similar_checked(M, topn, measure, queries=q)
        nrm = np.linalg.norm(M, axis=1)
        B = M / nrm[:, None] if measure == "cosine" else M
        for b0 in range(0, len(q), 64):
            qb = q[b0:b0 + 64]
            check_rows(ids[b0:b0 + 64], sc[b0:b0 + 64], B[qb], B, candidates(None, qb, n), topn)
        a_i, a_s = similar_checked(M, topn, measure, queries=q[::-1].copy())
        assert np.array_equal(a_i, ids[::-1]) and np.array_equal(bits(a_s), bits(sc[::-1]))


@gpu
def test_argument_errors():
    rng = np.random.default_rng(1)
    n, k = 300, 8
    M = rng.standard_normal((n, k))
    ex = random_exclusion(n, n, rng, 20)
    bad_id = Ratings(n, n, ex.row_ptr.copy(), ex.item.copy(), ex.rating)
    bad_id.item[5] = n
    desc = Ratings(n, n, ex.row_ptr.copy(), ex.item.copy(), ex.rating)
    a = int(desc.row_ptr[int(np.flatnonzero(np.diff(ex.row_ptr) >= 2)[0])])      # a row's ids are distinct: swap two
    desc.item[a], desc.item[a + 1] = desc.item[a + 1], desc.item[a]
    cases = [
        lambda: api.similar(M, 0),
        lambda: api.similar(M, 257),
        lambda: api.similar(rng.standard_normal((n, 257)), 5),
        lambda: api.similar(M, 5, queries=[0, n]),
        lambda: api.similar(M, 5, queries=[-1]),
        lambda: api.similar(M, 5, exclude=bad_id),
        lambda: api.similar(M, 5, exclude=desc),
        lambda: api.similar(M, 5, measure="jaccard"),
    ]
    for f in cases:
        with pytest.raises(api.PrimalCRError):
            f()
    L = api.lib()
    rp = np.ascontiguousarray(ex.row_ptr, np.int64); it = np.ascontiguousarray(ex.item, np.int32)
    q = np.arange(4, dtype=np.int32)
    out_i = np.empty((n, 5), np.int32); out_s = np.empty((n, 5))
    raw = [
        (M.ctypes.data, n, k, 7, rp.ctypes.data, it.ctypes.data, None, n, 5, out_i.ctypes.data, out_s.ctypes.data, 0),  # measure
        (M.ctypes.data, n, k, 1, rp.ctypes.data, None, None, n, 5, out_i.ctypes.data, out_s.ctypes.data, 0),  # ptr w/o ids
        (M.ctypes.data, n, k, 1, None, None, None, n, 5, None, out_s.ctypes.data, 0),                          # NULL ids_out
        (M.ctypes.data, n, k, 0, None, None, q.ctypes.data, 4, 5, None, None, 0),                              # NULL ids_out
        (M.ctypes.data, n, k, 1, None, None, None, n - 1, 5, out_i.ctypes.data, None, 0),                      # NULL queries
        (None, n, k, 1, None, None, None, n, 5, out_i.ctypes.data, None, 0),                                   # NULL M
        (M.ctypes.data, -1, k, 1, None, None, None, 0, 5, out_i.ctypes.data, None, 0),                          # n < 0
        (M.ctypes.data, n, 0, 1, None, None, None, n, 5, out_i.ctypes.data, None, 0),                          # k = 0
        (M.ctypes.data, n, k, 1, None, None, None, n, 5, out_i.ctypes.data, None, 99),                         # device
    ]
    for args in raw:
        assert L.primalcr_similar(*args) == -1, (args, L.primalcr_last_error())
    ids, sc = similar_checked(M, 5, "cosine", ex)       # a valid call afterwards
    B = M / np.linalg.norm(M, axis=1)[:, None]
    check_rows(ids, sc, B, B, candidates(ex, np.arange(n), n), 5)


@gpu
def test_cli_matches_api(tmp_path):
    assert os.path.exists(SIM), "run __graft_entry__.build()"
    rng = np.random.default_rng(9)
    U = rng.standard_normal((90, 12)); V = rng.standard_normal((400, 12))
    V[17] = 0.0                                         # NaN cosine scores in the output
    save_model(str(tmp_path / "model"), U, V)
    for side, M in (("items", V), ("users", U)):
        for measure in ("cosine", "dot"):
            for ids_in in (None, [5, 1, 5, 24, 13, 18]):
                args = [SIM, "-s", side, "-m", measure, "-n", "10"]
                if ids_in is not None:
                    (tmp_path / "ids").write_text("".join("%d\n" % u for u in ids_in))
                    args += ["-q", str(tmp_path / "ids")]
                r = subprocess.run(args + [str(tmp_path / "model"), str(tmp_path / "out")], capture_output=True, text=True)
                assert r.returncode == 0, r.stderr
                qi = None if ids_in is None else np.array(ids_in, np.int32) - 1
                it, sc = api.similar(M, 10, measure=measure, queries=qi)
                want_q = np.arange(1, M.shape[0] + 1) if ids_in is None else np.array(ids_in)
                lines = open(tmp_path / "out").read().split("\n")[:-1]
                want = ["%d %d %.17g" % (q, i + 1, s) for t, q in enumerate(want_q) for i, s in zip(it[t], sc[t]) if i >= 0]
                assert lines == want, (side, measure, ids_in)
                got = np.array([float(l.split()[2]) for l in lines])
                wnt = np.array([s for t in range(len(want_q)) for i, s in zip(it[t], sc[t]) if i >= 0])
                assert np.array_equal(bits(got), bits(wnt))     # %.17g round-trips the doubles (NaN as one NaN)
    # the defaults: items, cosine, top 10
    r = subprocess.run([SIM, str(tmp_path / "model"), str(tmp_path / "out")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    it, sc = api.similar(V, 10)
    assert open(tmp_path / "out").read().count("\n") == int((it >= 0).sum())
    # errors exit non-zero
    (tmp_path / "bad").write_text("401\n")
    for args in (["-s", "movies"], ["-m", "l2"], ["-n", "0"], ["-q", str(tmp_path / "bad")], ["-q", str(tmp_path / "none")]):
        r = subprocess.run([SIM] + args + [str(tmp_path / "model"), str(tmp_path / "out")], capture_output=True, text=True)
        assert r.returncode == 1, args
    r = subprocess.run([SIM, str(tmp_path / "nomodel"), str(tmp_path / "out")], capture_output=True, text=True)
    assert r.returncode == 1
