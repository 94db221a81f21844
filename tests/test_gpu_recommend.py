"""Top-N recommendation (primalcr_recommend / api.recommend / primalcr-recommend) against a numpy reference.

The reference scores U[users] @ V.T in user blocks, masks excluded items and orders each row by
(NaN last, score descending, item ascending) -- the library's total order."""
import os
import subprocess

import numpy as np
import pytest

from primalcr_b200 import api
from primalcr_b200.data import Ratings, save_model, synth_dataset, write_reference_dir
from tests.util import dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REC = os.path.join(ROOT, "primalcr_b200", "bin", "primalcr-recommend")


# ----------------------------------------------------------------------------- reference
def eligible(excl: Ratings | None, users, d2):
    ok = np.ones((len(users), d2), bool)
    if excl is not None:
        for r, u in enumerate(users):
            ok[r, excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]]] = False
    return ok


def ref_topn(S, ok, n, exact=True):
    """Items and scores of the n best eligible entries of every row of S, padded with -1 / NaN.  exact: the full total
    order (ties, NaN); otherwise argpartition + sort of the n survivors (finite scores, near ties are judged by check_rows)."""
    rows, d2 = S.shape
    m = min(n, d2)
    if exact:
        isn = np.isnan(S)
        neg = np.where(isn, 0.0, -S)
        it = np.broadcast_to(np.arange(d2), S.shape)
        order = np.lexsort((it, neg, isn, ~ok), axis=-1)[:, :m]
    else:
        neg = np.where(ok, -S, np.inf)
        part = np.argpartition(neg, m - 1, axis=1)[:, :m] if m < d2 else np.broadcast_to(np.arange(d2), S.shape).copy()
        order = np.take_along_axis(part, np.lexsort((part, np.take_along_axis(neg, part, 1)), axis=-1), 1)
    items = np.full((rows, n), -1, np.int32); scores = np.full((rows, n), np.nan)
    take = np.take_along_axis(ok, order, 1)
    items[:, :m] = np.where(take, order, -1)
    scores[:, :m] = np.where(take, np.take_along_axis(S, order, 1), np.nan)
    return items, scores


def check_rows(items, scores, Ub, V, ok, n, rel=1e-13, near=1e-12):
    """The rules for non-exact factors: scores equal U[u].V[i] to `rel`, rows non-increasing with no excluded or repeated
    item, the items equal the reference's except where reference scores within near*max|score| swap places, and nothing
    eligible that was left out beats the last returned score by more than that."""
    S = Ub @ V.T
    A = np.abs(Ub) @ np.abs(V).T
    cnt = np.minimum(ok.sum(1), n)
    pos = np.arange(n)[None, :]
    assert np.array_equal(items >= 0, pos < cnt[:, None])
    assert np.all(np.isnan(scores[items < 0]))
    r_idx = np.broadcast_to(np.arange(len(items))[:, None], items.shape)
    have = items >= 0
    it = np.where(have, items, 0)
    true = S[r_idx, it]
    err = np.abs(scores - true)[have]
    assert np.all(err <= rel * A[r_idx, it][have] + 1e-300), err.max()
    assert np.all(ok[r_idx, it][have])
    srt = np.sort(np.where(have, items, -1 - pos), axis=1)
    assert np.all(np.diff(srt, axis=1) != 0)
    assert np.all((np.diff(scores, axis=1) <= 0) | ~have[:, 1:])
    tol = near * np.max(np.abs(np.where(ok, S, 0.0)), axis=1, initial=0.0)[:, None]
    ri, rs = ref_topn(S, ok, n, exact=False)
    assert np.array_equal(ri >= 0, have)
    same = (ri == items) | (np.abs(rs - true) <= tol)
    assert np.all(same[have])
    left = ok.copy()
    left[r_idx[have], items[have]] = False
    best_left = np.max(np.where(left, S, -np.inf), axis=1)
    last = np.min(np.where(have, true, np.inf), axis=1)
    assert np.all(last >= best_left - tol[:, 0])


def recommend_checked(U, V, n, excl, users=None):
    it, sc = api.recommend(U, V, n, exclude=excl, users=users)
    us = np.arange(U.shape[0]) if users is None else np.asarray(users)
    assert it.shape == (len(us), n) and sc.shape == (len(us), n) and it.dtype == np.int32 and sc.dtype == np.float64
    return it, sc, us


def random_exclusion(d1, d2, rng, max_len):
    users, items = [], []
    for u in range(d1):
        m = int(rng.integers(0, max_len + 1))
        items.append(np.sort(rng.choice(d2, size=min(m, d2), replace=False))); users.append(np.full(len(items[-1]), u))
    return Ratings.from_coo(d1, d2, np.concatenate(users), np.concatenate(items), np.ones(sum(len(x) for x in items)))


# ----------------------------------------------------------------------------- CPU
def test_recommend_without_gpu_fails_loudly(have_gpu):
    if have_gpu:
        pytest.skip("a GPU is present")
    U = np.ones((3, 2)); V = np.ones((5, 2))
    with pytest.raises(api.PrimalCRError, match="no CPU fallback|CUDA"):
        api.recommend(U, V, 2)


# ----------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


@gpu
@pytest.mark.parametrize("with_excl", [False, True])
def test_exact_ties_match_reference(with_excl):
    rng = np.random.default_rng(11)
    d1, d2, k = 300, 700, 8
    U = rng.integers(-3, 4, size=(d1, k)).astype(np.float64)
    V = rng.integers(-3, 4, size=(d2, k)).astype(np.float64)
    U[[0, 17, 299]] = 0.0                       # all-zero scores: +0.0 and -0.0 must tie
    U[5] = -U[4]
    V[[3, 600]] = 0.0
    excl = random_exclusion(d1, d2, rng, 400) if with_excl else None
    excl_users = np.arange(d1)
    ok = eligible(excl, excl_users, d2)
    S = U @ V.T                                 # every product and sum is an exact integer
    for n in (1, 5, 37, 256):
        it, sc, _ = recommend_checked(U, V, n, excl)
        ri, rs = ref_topn(S, ok, n)
        assert np.array_equal(it, ri), n
        assert np.array_equal(sc, rs, equal_nan=True), n


@gpu
@pytest.mark.parametrize("k", [1, 7, 100, 256])
def test_random_factors_ml1m(k):
    ds = dataset("ml1m")
    rng = np.random.default_rng(100 + k)
    U = rng.standard_normal((ds.d1, k)); V = rng.standard_normal((ds.d2, k))
    ok = eligible(ds.train, np.arange(ds.d1), ds.d2)
    for n in (1, 10, 100, 256):
        it, sc, _ = recommend_checked(U, V, n, ds.train)
        check_rows(it, sc, U, V, ok, n)


@gpu
def test_ragged_edge_cases():
    ds = dataset("ragged")
    d1, d2, k = ds.d1, ds.d2, 10
    rng = np.random.default_rng(5)
    U = rng.standard_normal((d1, k)); V = rng.standard_normal((d2, k))
    full_i, full_s, _ = recommend_checked(U, V, 256, ds.train)      # 0-rating users, 4097 / 5000 of 6000 items excluded
    check_rows(full_i, full_s, U, V, eligible(ds.train, np.arange(d1), d2), 256)
    # fewer eligible items than topn: user 0 excludes every item, user 1 all but seven
    us, its = [np.zeros(d2, int), np.ones(d2 - 7, int)], [np.arange(d2), np.arange(7, d2)]
    ex = Ratings.from_coo(d1, d2, np.concatenate(us), np.concatenate(its), np.ones(2 * d2 - 7))
    it, sc, _ = recommend_checked(U, V, 20, ex)
    assert np.all(it[0] == -1) and np.all(np.isnan(sc[0]))
    assert np.all(it[1, 7:] == -1) and np.all(np.isnan(sc[1, 7:])) and sorted(it[1, :7]) == list(range(7))
    check_rows(it, sc, U, V, eligible(ex, np.arange(d1), d2), 20)
    # d2 < topn
    V50 = V[:50].copy()
    it, sc, _ = recommend_checked(U, V50, 100, None)
    assert np.all(it[:, 50:] == -1) and np.all(np.isnan(sc[:, 50:]))
    check_rows(it, sc, U, V50, np.ones((d1, 50), bool), 100)
    # a user subset in arbitrary order with repeats: the same rows, bit for bit
    sub = np.array([20, 3, 3, 0, 23, 19, 20, 18], np.int32)
    it, sc, _ = recommend_checked(U, V, 256, ds.train, users=sub)
    assert np.array_equal(it, full_i[sub]) and np.array_equal(sc.view(np.int64), full_s[sub].view(np.int64))
    # n_users = 0
    it, sc, _ = recommend_checked(U, V, 5, ds.train, users=np.zeros(0, np.int32))
    assert it.shape == (0, 5)
    # exclude=None
    it, sc, _ = recommend_checked(U, V, 64, None)
    check_rows(it, sc, U, V, np.ones((d1, d2), bool), 64)


@gpu
def test_nan_user_and_nan_item():
    rng = np.random.default_rng(21)
    d1, d2, k, n = 200, 3000, 16, 40
    U = rng.standard_normal((d1, k)); V = rng.standard_normal((d2, k))
    U[7] = np.nan; V[11] = np.nan
    excl = random_exclusion(d1, d2, rng, 50)
    ok = eligible(excl, np.arange(d1), d2)
    it, sc, _ = recommend_checked(U, V, n, excl)
    assert np.array_equal(it[7], np.flatnonzero(ok[7])[:n]) and np.all(np.isnan(sc[7]))
    others = np.arange(d1) != 7
    assert not np.any(it[others] == 11)
    assert np.all(np.isfinite(sc[others]))
    # the NaN item ranks after every finite item: with topn = d2 it is the last eligible entry
    it2, sc2, _ = recommend_checked(U[:3], V, 256, None)
    V2 = V[:200].copy()
    it3, sc3, _ = recommend_checked(U[:3], V2, 256, None)
    assert np.all(it3[:, 199] == 11) and np.all(np.isnan(sc3[:, 199])) and np.all(it3[:, 200:] == -1)
    assert not np.any(it2 == 11)
    # the device is still usable
    it4, _, _ = recommend_checked(U[:10], V, 5, None)
    assert np.all(it4[:7] >= 0)


@gpu
def test_deterministic_and_batch_independent():
    ds = dataset("ml1m")
    rng = np.random.default_rng(3)
    U = rng.standard_normal((ds.d1, 100)); V = rng.standard_normal((ds.d2, 100))
    a_i, a_s, _ = recommend_checked(U, V, 100, ds.train)
    b_i, b_s, _ = recommend_checked(U, V, 100, ds.train)
    assert np.array_equal(a_i, b_i) and np.array_equal(a_s.view(np.int64), b_s.view(np.int64))
    sub = rng.choice(ds.d1, size=500, replace=True).astype(np.int32)
    c_i, c_s, _ = recommend_checked(U, V, 100, ds.train, users=sub)
    assert np.array_equal(c_i, a_i[sub]) and np.array_equal(c_s.view(np.int64), a_s[sub].view(np.int64))
    for u in (0, 1, 4321, ds.d1 - 1):
        d_i, d_s, _ = recommend_checked(U, V, 100, ds.train, users=[u])
        assert np.array_equal(d_i[0], a_i[u]) and np.array_equal(d_s[0].view(np.int64), a_s[u].view(np.int64))


@gpu
def test_netflix_shape_scale():
    ds = synth_dataset("netflix", scale=0.05, test_per_user=0)
    k, n = 100, 100
    rng = np.random.default_rng(7)
    U = rng.standard_normal((ds.d1, k)); V = rng.standard_normal((ds.d2, k))
    it, sc, _ = recommend_checked(U, V, n, ds.train)
    for b0 in range(0, ds.d1, 1024):
        us = np.arange(b0, min(ds.d1, b0 + 1024))
        check_rows(it[us], sc[us], U[us], V, eligible(ds.train, us, ds.d2), n)


@gpu
def test_argument_errors():
    ds = dataset("ragged")
    rng = np.random.default_rng(1)
    U = rng.standard_normal((ds.d1, 8)); V = rng.standard_normal((ds.d2, 8))
    bad_item = Ratings(ds.d1, ds.d2, ds.train.row_ptr.copy(), ds.train.item.copy(), ds.train.rating)
    bad_item.item[5] = ds.d2
    desc = Ratings(ds.d1, ds.d2, ds.train.row_ptr.copy(), ds.train.item.copy(), ds.train.rating)
    a = int(desc.row_ptr[10]); desc.item[a], desc.item[a + 1] = desc.item[a + 1], desc.item[a]
    cases = [
        lambda: api.recommend(U, V, 0),
        lambda: api.recommend(U, V, 257),
        lambda: api.recommend(rng.standard_normal((ds.d1, 257)), rng.standard_normal((ds.d2, 257)), 5),
        lambda: api.recommend(U, V, 5, users=[0, ds.d1]),
        lambda: api.recommend(U, V, 5, exclude=bad_item),
        lambda: api.recommend(U, V, 5, exclude=desc),
    ]
    for f in cases:
        with pytest.raises(api.PrimalCRError):
            f()
    L = api.lib()
    rp = np.ascontiguousarray(ds.train.row_ptr, np.int64)
    out_i = np.empty((ds.d1, 5), np.int32); out_s = np.empty((ds.d1, 5))
    rc = L.primalcr_recommend(U.ctypes.data, ds.d1, V.ctypes.data, ds.d2, 8, rp.ctypes.data, None, None, ds.d1, 5,
                              out_i.ctypes.data, out_s.ctypes.data, 0)
    assert rc == -1, L.primalcr_last_error()
    it, sc = api.recommend(U, V, 5, exclude=ds.train)       # a valid call afterwards
    check_rows(it, sc, U, V, eligible(ds.train, np.arange(ds.d1), ds.d2), 5)


@gpu
def test_cli_matches_api(tmp_path):
    assert os.path.exists(REC), "run __graft_entry__.build()"
    ds = dataset("ragged")
    rng = np.random.default_rng(9)
    U = rng.standard_normal((ds.d1, 12)); V = rng.standard_normal((ds.d2, 12))
    write_reference_dir(str(tmp_path / "data"), ds)
    save_model(str(tmp_path / "model"), U, V)
    for users in (None, [5, 1, 5, 24, 13]):
        args = [REC, "-n", "10", "-e", str(tmp_path / "data")]
        if users is not None:
            (tmp_path / "users").write_text("".join("%d\n" % u for u in users))
            args += ["-u", str(tmp_path / "users")]
        r = subprocess.run(args + [str(tmp_path / "model"), str(tmp_path / "out")], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        ui = None if users is None else np.array(users, np.int32) - 1
        it, sc = api.recommend(U, V, 10, exclude=ds.train, users=ui)
        want_users = np.arange(1, ds.d1 + 1) if users is None else np.array(users)
        lines = open(tmp_path / "out").read().split("\n")[:-1]
        want = ["%d %d %.17g" % (u, i + 1, s) for q, u in enumerate(want_users) for i, s in zip(it[q], sc[q]) if i >= 0]
        assert lines == want
        got = [tuple(map(float, l.split())) for l in lines]
        wnt = [(float(u), float(i + 1), s) for q, u in enumerate(want_users) for i, s in zip(it[q], sc[q]) if i >= 0]
        assert got == wnt                       # %.17g round-trips the doubles
    save_model(str(tmp_path / "model2"), np.vstack([U, U[:1]]), V)
    r = subprocess.run([REC, "-n", "10", "-e", str(tmp_path / "data"), str(tmp_path / "model2"), str(tmp_path / "out2")],
                       capture_output=True, text=True)
    assert r.returncode != 0
