"""Held-out ranking evaluation (primalcr_rank_heldout / primalcr_rank_metrics, api.heldout_ranks / api.ranking_metrics,
primalcr-rankeval).

Ranks are checked against a numpy reference that counts, for every held-out entry, the eligible items that beat it under
the library's total order (score descending, item ascending, +0.0 == -0.0, NaN last), and against api.recommend: an entry
of rank r <= 256 sits at position r-1 of the user's top-256 row with the same score bit for bit.  The metrics are checked
against a plain numpy restatement of their definitions."""
import math
import os
import subprocess

import numpy as np
import pytest

from primalcr_b200 import api
from primalcr_b200.data import Ratings, csr_in_file_order, save_model, synth_dataset, write_reference_dir
from tests.util import dataset

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RANKEVAL = os.path.join(ROOT, "primalcr_b200", "bin", "primalcr-rankeval")


# ----------------------------------------------------------------------------- references
def ref_ranks(S, heldout: Ratings, excl: Ratings | None):
    """1 + the number of eligible items better than each held-out entry; 0 for an excluded item."""
    d2 = S.shape[1]
    ids = np.arange(d2)
    out = np.zeros(heldout.nnz, np.int64)
    for u in range(heldout.d1):
        a, b = int(heldout.row_ptr[u]), int(heldout.row_ptr[u + 1])
        if a == b:
            continue
        ok = np.ones(d2, bool)
        if excl is not None:
            ok[excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]]] = False
        s = S[u]
        nan = np.isnan(s)
        for e in range(a, b):
            i = int(heldout.item[e])
            if not ok[i]:
                continue
            if nan[i]:
                bt = ~nan | (nan & (ids < i))
            else:
                bt = (~nan & (s > s[i])) | ((s == s[i]) & (ids < i))
            out[e] = 1 + int(np.count_nonzero(bt & ok))
    return out


def ref_metrics(d2, excl, heldout, rank, cutoffs, min_rating):
    """The definitions of primalcr_rank_metrics, restated per user."""
    acc = {("recall", n): [] for n in cutoffs}
    acc.update({("precision", n): [] for n in cutoffs}); acc.update({("ndcg", n): [] for n in cutoffs})
    mrr, auc = [], []
    for u in range(heldout.d1):
        a, b = int(heldout.row_ptr[u]), int(heldout.row_ptr[u + 1])
        items = {}
        for e in range(a, b):
            if rank[e] > 0:
                i = int(heldout.item[e])
                r0, k0 = items.get(i, (-np.inf, np.inf))
                items[i] = (max(r0, heldout.rating[e]), min(k0, int(rank[e])))
        rel = sorted(k for r, k in items.values() if r >= min_rating)
        if not rel:
            continue
        for n in cutoffs:
            hits = [k for k in rel if k <= n]
            acc[("recall", n)].append(len(hits) / len(rel))
            acc[("precision", n)].append(len(hits) / n)
            dcg = sum(1.0 / math.log2(k + 1) for k in hits)
            idcg = sum(1.0 / math.log2(p + 1) for p in range(1, min(n, len(rel)) + 1))
            acc[("ndcg", n)].append(dcg / idcg)
        mrr.append(1.0 / rel[0])
        cand = d2 - (len(np.unique(excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]])) if excl is not None else 0)
        nn = cand - len(rel)
        if nn > 0:
            auc.append(sum(nn - (k - 1 - sum(1 for q in rel if q < k)) for k in rel) / (len(rel) * nn))
    out = {"%s@%d" % key: float(np.mean(v)) if v else math.nan for key, v in acc.items()}
    out.update(mrr=float(np.mean(mrr)) if mrr else math.nan, auc=float(np.mean(auc)) if auc else math.nan, n_users=len(mrr))
    return out


def close(got, want, rel=1e-12):
    assert set(got) == set(want), (sorted(got), sorted(want))
    for key in want:
        g, w = got[key], want[key]
        if isinstance(w, float) and math.isnan(w):
            assert math.isnan(g), key
        else:
            assert abs(g - w) <= rel * abs(w) + 1e-300, (key, g, w)


def heldout_of(d1, d2, rows):
    """File-order held-out CSR from {user: [(item, rating), ...]}."""
    rows = sorted(rows.items())
    us = [u for u, ent in rows for _ in ent]
    it = [i for _, ent in rows for i, _ in ent]
    rt = [r for _, ent in rows for _, r in ent]
    return csr_in_file_order(d1, d2, np.array(us, np.int64), np.array(it, np.int64), np.array(rt, np.float64))


def random_exclusion(d1, d2, rng, max_len):
    users, items = [], []
    for u in range(d1):
        m = int(rng.integers(0, max_len + 1))
        items.append(np.sort(rng.choice(d2, size=min(m, d2), replace=False))); users.append(np.full(len(items[-1]), u))
    return Ratings.from_coo(d1, d2, np.concatenate(users), np.concatenate(items), np.ones(sum(len(x) for x in items)))


def random_heldout(d1, d2, rng, max_len, excl=None, overlap=0, min_len=0):
    """min_len to max_len distinct held-out items per user in random (file) order, disjoint from excl except for `overlap`
    excluded items per user."""
    rows = {}
    for u in range(d1):
        ex = set() if excl is None else set(excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]].tolist())
        free = np.array([i for i in range(d2) if i not in ex])
        m = min(int(rng.integers(min_len, max_len + 1)), len(free))
        take = rng.choice(free, size=m, replace=False).tolist()
        if overlap and ex:
            take += rng.choice(sorted(ex), size=min(overlap, len(ex)), replace=False).tolist()
        rng.shuffle(take)
        rows[u] = [(int(i), float(rng.integers(1, 6))) for i in take]
    return heldout_of(d1, d2, rows)


# ----------------------------------------------------------------------------- CPU: metrics
def metric_case():
    """Hand-built ranks: duplicates with different ratings, rank-0 entries, users with no relevant item, a user whose
    relevant items fill all its candidates, exclusion rows with repeats."""
    d1, d2 = 7, 12
    excl = Ratings(d1, d2, np.array([0, 3, 3, 6, 6, 18, 18, 20], np.int64),
                   np.array([1, 1, 4, 0, 2, 2] + list(range(12)) + [3, 3], np.int32), np.ones(20))
    # (item, rating, rank) per user, file order
    rows = {
        0: [(5, 4.0, 3), (7, 2.0, 1), (5, 5.0, 3), (1, 5.0, 0), (9, 3.0, 10)],   # item 5 twice, item 1 excluded: rank 0
        1: [(0, 1.0, 2), (3, 2.0, 5)],                                           # nothing >= 3: not evaluated at min 3
        2: [(3, 5.0, 1), (4, 4.0, 2), (6, 1.0, 7)],
        3: [(2, 4.0, 0)],                                                        # only a rank-0 entry
        4: [],                                                                   # everything excluded
        5: [(0, 5.0, 1), (1, 5.0, 2), (2, 4.5, 3), (4, 4.0, 4), (5, 3.0, 5), (6, 5.0, 6), (7, 5.0, 7), (8, 5.0, 8),
            (9, 5.0, 9), (10, 5.0, 10), (11, 5.0, 11), (1, 3.0, 2), (3, 5.0, 12)],  # relevant = all 12 candidates
        6: [(11, -2.5, 4), (0, 0.5, 12)],                                        # real-valued / negative ratings
    }
    ho = heldout_of(d1, d2, {u: [(i, r) for i, r, _ in ent] for u, ent in rows.items()})
    rank = np.zeros(ho.nnz, np.int32)
    for u, ent in rows.items():            # csr_in_file_order keeps file order inside a user
        rank[ho.row_ptr[u]:ho.row_ptr[u + 1]] = [k for _, _, k in ent]
    return d2, excl, ho, rank


@pytest.mark.parametrize("min_rating", [None, 3.0, 1.0])
def test_metrics_match_definitions(min_rating):
    d2, excl, ho, rank = metric_case()
    cutoffs = (1, 3, 5, 10, 100)                         # 100 > d2
    got = api.ranking_metrics(rank, ho, exclude=excl, cutoffs=cutoffs, min_rating=min_rating)
    want = ref_metrics(d2, excl, ho, rank, cutoffs, -np.inf if min_rating is None else min_rating)
    close(got, want)
    assert got["n_users"] == (5 if min_rating is None else 4 if min_rating == 1.0 else 3)


def test_metrics_random_against_definitions():
    rng = np.random.default_rng(4)
    d1, d2 = 60, 50
    excl = random_exclusion(d1, d2, rng, 20)
    ho = random_heldout(d1, d2, rng, 15, excl=excl, overlap=1)
    rank = rng.integers(0, d2 + 1, size=ho.nnz).astype(np.int32)
    for min_rating in (None, 4.0):
        got = api.ranking_metrics(rank, ho, exclude=excl, cutoffs=(2, 20, 60), min_rating=min_rating)
        close(got, ref_metrics(d2, excl, ho, rank, (2, 20, 60), -np.inf if min_rating is None else min_rating))
    got = api.ranking_metrics(rank, ho, cutoffs=(5,))    # nothing excluded: C_u = d2
    close(got, ref_metrics(d2, None, ho, rank, (5,), -np.inf))


def test_metrics_no_user_is_nan():
    d2, excl, ho, rank = metric_case()
    got = api.ranking_metrics(np.zeros_like(rank), ho, exclude=excl, cutoffs=(10,))
    assert got["n_users"] == 0 and all(math.isnan(got[k]) for k in ("recall@10", "ndcg@10", "mrr", "auc"))


def test_metrics_argument_errors():
    d2, excl, ho, rank = metric_case()
    bad_rank = rank.copy(); bad_rank[0] = d2 + 1
    neg_rank = rank.copy(); neg_rank[1] = -1
    bad_item = Ratings(ho.d1, ho.d2, ho.row_ptr.copy(), ho.item.copy(), ho.rating); bad_item.item[2] = d2
    bad_ptr = Ratings(ho.d1, ho.d2, ho.row_ptr.copy(), ho.item, ho.rating); bad_ptr.row_ptr[2] = bad_ptr.row_ptr[1] - 1
    bad_first = Ratings(ho.d1, ho.d2, ho.row_ptr.copy(), ho.item, ho.rating); bad_first.row_ptr[0] = 1
    desc = Ratings(excl.d1, excl.d2, excl.row_ptr.copy(), excl.item.copy(), excl.rating); desc.item[[0, 2]] = desc.item[[2, 0]]
    cases = [
        lambda: api.ranking_metrics(bad_rank, ho, exclude=excl),
        lambda: api.ranking_metrics(neg_rank, ho, exclude=excl),
        lambda: api.ranking_metrics(rank, ho, exclude=excl, cutoffs=(10, 0)),
        lambda: api.ranking_metrics(rank, bad_item, exclude=excl),
        lambda: api.ranking_metrics(rank, bad_ptr, exclude=excl),
        lambda: api.ranking_metrics(rank, bad_first, exclude=excl),
        lambda: api.ranking_metrics(rank, ho, exclude=desc),
    ]
    for f in cases:
        with pytest.raises(api.PrimalCRError, match="error -1"):
            f()
    L = api.lib()
    rp = np.ascontiguousarray(excl.row_ptr, np.int64)
    rc = L.primalcr_rank_metrics(ho.d1, d2, rp.ctypes.data, None, ho.row_ptr.ctypes.data, ho.item.ctypes.data,
                                 ho.rating.ctypes.data, rank.ctypes.data, 0.0, None, 0, None, None, None, None, None, None)
    assert rc == -1
    rc = L.primalcr_rank_metrics(ho.d1, d2, None, None, ho.row_ptr.ctypes.data, None, ho.rating.ctypes.data,
                                 rank.ctypes.data, 0.0, None, 0, None, None, None, None, None, None)
    assert rc == -1
    close(api.ranking_metrics(rank, ho, exclude=excl), ref_metrics(d2, excl, ho, rank, (10,), -np.inf))


def test_heldout_ranks_without_gpu_fails_loudly(have_gpu):
    if have_gpu:
        pytest.skip("a GPU is present")
    U = np.ones((3, 2)); V = np.ones((5, 2))
    ho = heldout_of(3, 5, {0: [(1, 1.0)], 2: [(4, 2.0)]})
    with pytest.raises(api.PrimalCRError, match="no CPU fallback|CUDA"):
        api.heldout_ranks(U, V, ho)


# ----------------------------------------------------------------------------- GPU
gpu = pytest.mark.gpu


def ranks_checked(U, V, ho, excl):
    r, s = api.heldout_ranks(U, V, ho, exclude=excl)
    assert r.dtype == np.int32 and s.dtype == np.float64 and r.shape == (ho.nnz,) and s.shape == (ho.nnz,)
    return r, s


def check_against_recommend(U, V, ho, excl, r, s, users=None, n=256):
    """Rank r <= n: position r-1 of recommend's row, same score bits; r > n: not in the row; r == 0: excluded."""
    users = np.arange(ho.d1) if users is None else np.asarray(users)
    it, sc = api.recommend(U, V, n, exclude=excl, users=users.astype(np.int32))
    for q, u in enumerate(users):
        a, b = int(ho.row_ptr[u]), int(ho.row_ptr[u + 1])
        ex = set() if excl is None else set(excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]].tolist())
        row = it[q].tolist()
        for e in range(a, b):
            i, k = int(ho.item[e]), int(r[e])
            if k == 0:
                assert i in ex, (u, i)
                continue
            assert i not in ex, (u, i)
            if k <= n:
                assert row[k - 1] == i, (u, i, k)
                assert sc[q, k - 1].view(np.int64) == s[e].view(np.int64), (u, i, k)
            else:
                assert i not in row, (u, i, k)


@gpu
@pytest.mark.parametrize("with_excl", [False, True])
def test_exact_ties_match_reference(with_excl):
    rng = np.random.default_rng(12)
    d1, d2, k = 150, 900, 8
    U = rng.integers(-3, 4, size=(d1, k)).astype(np.float64)
    V = rng.integers(-3, 4, size=(d2, k)).astype(np.float64)
    U[[0, 17]] = 0.0                          # all-zero users and items: long runs of exact ties at 0.0
    U[5] = -U[4]
    V[[3, 600]] = 0.0
    U[9] = np.nan                             # a NaN user: every score NaN, ties decided by item id
    V[11] = np.nan                            # a NaN item: last for every user
    excl = random_exclusion(d1, d2, rng, 300) if with_excl else None
    ho = random_heldout(d1, d2, rng, 40, excl=excl, overlap=2, min_len=1)
    S = U @ V.T                               # every product and sum is an exact integer
    r, s = ranks_checked(U, V, ho, excl)
    assert np.array_equal(r, ref_ranks(S, ho, excl))
    # the NaN user: 1 + the eligible items with a smaller id
    a, b = int(ho.row_ptr[9]), int(ho.row_ptr[10])
    ok = np.ones(d2, bool)
    if excl is not None:
        ok[excl.item[excl.row_ptr[9]:excl.row_ptr[10]]] = False
    for e in range(a, b):
        i = int(ho.item[e])
        assert r[e] == (1 + np.count_nonzero(ok[:i]) if ok[i] else 0)
    check_against_recommend(U, V, ho, excl, r, s)


@gpu
def test_signed_zero_scores_tie():
    """-0.0 scores: fma(1e-200, -1e-200, +0.0) rounds the exact -1e-400 to -0.0, and the other columns add 0 * -0.0 = -0.0,
    so the chain keeps it (k = 8 is a whole k chunk: no zero padding turns it into +0.0).  -0.0 ties with +0.0 and the item
    id decides; scores come back as primalcr_recommend returns them, +0.0."""
    rng = np.random.default_rng(31)
    d1, d2, k = 4, 700, 8
    U = np.zeros((d1, k)); U[:, 0] = [1e-200, -1e-200, 1.0, 0.0]
    V = np.full((d2, k), -0.0)
    V[:, 0] = rng.choice([1e-200, -1e-200, 0.0, -0.0, 1.0, -1.0], size=d2)
    S = U @ V.T                               # exact up to the sign of zero, which the reference ignores
    for excl in (None, random_exclusion(d1, d2, rng, 200)):
        ho = random_heldout(d1, d2, rng, 300, excl=excl, overlap=3, min_len=100)
        r, s = ranks_checked(U, V, ho, excl)
        assert np.array_equal(r, ref_ranks(S, ho, excl))
        assert not np.any((s == 0) & np.signbit(s))
        check_against_recommend(U, V, ho, excl, r, s)


@gpu
@pytest.mark.parametrize("k", [1, 7, 100, 256])
def test_agrees_with_recommend_ml1m(k):
    ds = dataset("ml1m")
    rng = np.random.default_rng(200 + k)
    U = rng.standard_normal((ds.d1, k)); V = rng.standard_normal((ds.d2, k))
    assert ds.test.nnz > 0
    r, s = ranks_checked(U, V, ds.test, ds.train)
    assert np.all((r >= 1) & (r <= ds.d2))    # the synthetic test set is disjoint from the training set
    check_against_recommend(U, V, ds.test, ds.train, r, s)


@gpu
def test_whole_rows_are_permutations():
    ds = dataset("ragged")                    # d2 = 6000; user 20 rates 5000 items, user 19 rates 4097
    d1, d2, k = ds.d1, ds.d2, 12
    rng = np.random.default_rng(8)
    U = rng.standard_normal((d1, k)); V = rng.standard_normal((d2, k))
    excl = ds.train
    rows = {}
    # user 20: every candidate (1000 items) plus 4000 excluded ones -> 5000 entries, 79 units
    ex20 = excl.item[excl.row_ptr[20]:excl.row_ptr[21]]
    cand20 = np.setdiff1d(np.arange(d2), ex20)
    rows[20] = [(int(i), 1.0) for i in rng.permutation(np.concatenate([cand20, ex20[:4000]]))]
    # user 4 (no training ratings): every item of the catalog
    rows[4] = [(int(i), 1.0) for i in rng.permutation(d2)]
    ho = heldout_of(d1, d2, rows)
    r, s = ranks_checked(U, V, ho, excl)
    a, b = int(ho.row_ptr[20]), int(ho.row_ptr[21])
    in_ex = np.isin(ho.item[a:b], ex20)
    assert np.all(r[a:b][in_ex] == 0)
    assert np.array_equal(np.sort(r[a:b][~in_ex]), np.arange(1, len(cand20) + 1))
    a, b = int(ho.row_ptr[4]), int(ho.row_ptr[5])
    assert np.array_equal(np.sort(r[a:b]), np.arange(1, d2 + 1))
    # the order the ranks give is the order of the scores
    order = np.argsort(r[a:b])
    sc = s[a:b][order]
    assert np.all(np.diff(sc) <= 0)
    check_against_recommend(U, V, ho, excl, r, s, users=[4, 20])


@gpu
def test_repeats_and_overlaps():
    rng = np.random.default_rng(3)
    d1, d2, k = 40, 2500, 16
    U = rng.standard_normal((d1, k)); V = rng.standard_normal((d2, k))
    excl = random_exclusion(d1, d2, rng, 100)
    rows = {}
    for u in range(d1):
        ex = excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]]
        free = np.setdiff1d(np.arange(d2), ex)
        base = rng.choice(free, size=30, replace=False).tolist()
        take = base + base[:7] + base[3:5] + (ex[:3].tolist() if len(ex) else [])   # repeats, excluded items
        rng.shuffle(take)
        rows[u] = [(int(i), 1.0) for i in take]
    ho = heldout_of(d1, d2, rows)
    r, s = ranks_checked(U, V, ho, excl)
    for u in range(d1):
        a, b = int(ho.row_ptr[u]), int(ho.row_ptr[u + 1])
        ex = set(excl.item[excl.row_ptr[u]:excl.row_ptr[u + 1]].tolist())
        seen = {}
        for e in range(a, b):
            i = int(ho.item[e])
            assert (r[e] == 0) == (i in ex)
            if i in seen:
                assert r[e] == r[seen[i]] and s[e].view(np.int64) == s[seen[i]].view(np.int64)
            seen[i] = e
    check_against_recommend(U, V, ho, excl, r, s)


@gpu
def test_deterministic_and_batch_independent():
    ds = dataset("ml1m")
    rng = np.random.default_rng(5)
    U = rng.standard_normal((ds.d1, 100)); V = rng.standard_normal((ds.d2, 100))
    r1, s1 = ranks_checked(U, V, ds.test, ds.train)
    r2, s2 = ranks_checked(U, V, ds.test, ds.train)
    assert np.array_equal(r1, r2) and np.array_equal(s1.view(np.int64), s2.view(np.int64))
    T = ds.test
    for u in (0, 17, ds.d1 - 1):
        a, b = int(T.row_ptr[u]), int(T.row_ptr[u + 1])
        if a == b:
            continue
        rp = np.zeros(ds.d1 + 1, np.int64); rp[u + 1:] = b - a
        one = Ratings(ds.d1, ds.d2, rp, T.item[a:b].copy(), T.rating[a:b].copy())
        r, s = ranks_checked(U, V, one, ds.train)
        assert np.array_equal(r, r1[a:b]) and np.array_equal(s.view(np.int64), s1[a:b].view(np.int64))


@gpu
def test_netflix_shape_scale():
    ds = synth_dataset("netflix", scale=0.05)
    k = 100
    rng = np.random.default_rng(7)
    U = rng.standard_normal((ds.d1, k)); V = rng.standard_normal((ds.d2, k))
    r, s = ranks_checked(U, V, ds.test, ds.train)
    assert ds.test.nnz > 0 and np.all((r >= 1) & (r <= ds.d2))
    users = np.sort(rng.choice(ds.d1, size=600, replace=False))
    check_against_recommend(U, V, ds.test, ds.train, r, s, users=users)


@gpu
def test_argument_errors():
    ds = dataset("ragged")
    rng = np.random.default_rng(1)
    U = rng.standard_normal((ds.d1, 8)); V = rng.standard_normal((ds.d2, 8))
    T = ds.test
    bad_item = Ratings(T.d1, T.d2, T.row_ptr.copy(), T.item.copy(), T.rating); bad_item.item[3] = ds.d2
    neg_item = Ratings(T.d1, T.d2, T.row_ptr.copy(), T.item.copy(), T.rating); neg_item.item[4] = -1
    dec = Ratings(T.d1, T.d2, T.row_ptr.copy(), T.item, T.rating); dec.row_ptr[3] = dec.row_ptr[2] - 1
    first = Ratings(T.d1, T.d2, T.row_ptr.copy(), T.item, T.rating); first.row_ptr[0] = 1
    desc = Ratings(ds.d1, ds.d2, ds.train.row_ptr.copy(), ds.train.item.copy(), ds.train.rating)
    a = int(desc.row_ptr[10]); desc.item[a], desc.item[a + 1] = desc.item[a + 1], desc.item[a]
    ex_item = Ratings(ds.d1, ds.d2, ds.train.row_ptr.copy(), ds.train.item.copy(), ds.train.rating)
    ex_item.item[-1] = ds.d2
    cases = [
        lambda: api.heldout_ranks(U, V, bad_item, exclude=ds.train),
        lambda: api.heldout_ranks(U, V, neg_item, exclude=ds.train),
        lambda: api.heldout_ranks(U, V, dec, exclude=ds.train),
        lambda: api.heldout_ranks(U, V, first, exclude=ds.train),
        lambda: api.heldout_ranks(U, V, T, exclude=desc),
        lambda: api.heldout_ranks(U, V, T, exclude=ex_item),
        lambda: api.heldout_ranks(rng.standard_normal((ds.d1, 257)), rng.standard_normal((ds.d2, 257)), T),
    ]
    for f in cases:
        with pytest.raises(api.PrimalCRError, match="error -1"):
            f()
    L = api.lib()
    out = np.empty(T.nnz, np.int32)
    rp = np.ascontiguousarray(ds.train.row_ptr, np.int64)
    calls = [   # NULL ho_row_ptr, NULL ho_item, NULL rank_out, excl_row_ptr without excl_item
        (None, T.item.ctypes.data, out.ctypes.data, None),
        (T.row_ptr.ctypes.data, None, out.ctypes.data, None),
        (T.row_ptr.ctypes.data, T.item.ctypes.data, None, None),
        (T.row_ptr.ctypes.data, T.item.ctypes.data, out.ctypes.data, rp.ctypes.data),
    ]
    for hp, hi, ro, ep in calls:
        rc = L.primalcr_rank_heldout(U.ctypes.data, ds.d1, V.ctypes.data, ds.d2, 8, ep, None, hp, hi, ro, None, 0)
        assert rc == -1, L.primalcr_last_error()
    r, s = ranks_checked(U, V, T, ds.train)             # a valid call afterwards
    check_against_recommend(U, V, T, ds.train, r, s)


@gpu
def test_cli_matches_api(tmp_path):
    assert os.path.exists(RANKEVAL), "run __graft_entry__.build()"
    ds = dataset("ragged")
    rng = np.random.default_rng(9)
    U = rng.standard_normal((ds.d1, 12)); V = rng.standard_normal((ds.d2, 12))
    write_reference_dir(str(tmp_path / "data"), ds)
    save_model(str(tmp_path / "model"), U, V)
    loaded = api.load_dir(str(tmp_path / "data"))
    for args, cutoffs, min_rating in (([], (10,), None), (["-n", "1,5,20,7000", "-r", "3"], (1, 5, 20, 7000), 3.0)):
        p = subprocess.run([RANKEVAL] + args + [str(tmp_path / "data"), str(tmp_path / "model")], capture_output=True,
                           text=True)
        assert p.returncode == 0, p.stderr
        r, _ = api.heldout_ranks(U, V, loaded.test, exclude=loaded.train)
        want = api.ranking_metrics(r, loaded.test, exclude=loaded.train, cutoffs=cutoffs, min_rating=min_rating)
        lines = p.stdout.split("\n")[:-1]
        assert lines == ["%s %.17g" % (key, v) if key != "n_users" else "n_users %d" % v for key, v in want.items()]
        assert want["n_users"] > 0
    save_model(str(tmp_path / "model2"), np.vstack([U, U[:1]]), V)
    p = subprocess.run([RANKEVAL, str(tmp_path / "data"), str(tmp_path / "model2")], capture_output=True, text=True)
    assert p.returncode != 0
    nodir = tmp_path / "notest"
    os.makedirs(nodir)
    write_reference_dir(str(nodir), ds)
    meta = (nodir / "meta").read_text().split("\n")
    (nodir / "meta").write_text("\n".join(meta[:2]) + "\n")
    p = subprocess.run([RANKEVAL, str(nodir), str(tmp_path / "model")], capture_output=True, text=True)
    assert p.returncode != 0 and "no test set" in p.stderr
