"""Scores loaded with set_scores stand in for the scores of the current factors in every call until the factors or the
scores change: update_V consumes them whether or not a read (here objective()) has built the sorted state from them
first, so the training that follows is bit-identical either way."""
import numpy as np
import pytest

from primalcr_b200 import api
from tests.util import dataset, init_factors, np_init

gpu = pytest.mark.gpu

K, LAM = 7, 50.0


def same_bits(a, b):
    return np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


def loaded_run(solver, m, read_first):
    """set_scores(m), optionally objective(), then update_V and update_U: objective, counters and factors after each."""
    ds = dataset("tiny")
    U, V = init_factors(ds.d1, ds.d2, K)
    e = api.Engine(api.Parameter(solver_type=solver, k=K, lambda_=LAM, maxiter=1))
    e.set_levels(np.unique(np.rint(ds.train.rating).astype(np.int64)))
    e.set_train(ds.train); e.set_factors(U, V)
    if m is not None:
        e.set_scores(m)
    if read_first:
        e.objective()
    out = []
    for step in (e.update_V, e.update_U):
        o = step()
        out.append((o, e.counters(), *e.get_factors()))
    e.close()
    return out


@gpu
@pytest.mark.parametrize("solver", [2, 1])
def test_loaded_scores_feed_update_V(solver):
    ds = dataset("tiny")
    P, Q = np_init(ds.d1, ds.d2, K, seed=5, scale=0.5)   # scores of other factors than the engine's
    users = np.repeat(np.arange(ds.d1), np.diff(ds.train.row_ptr))
    m = np.einsum("ij,ij->i", P[users], Q[ds.train.item])
    got = loaded_run(solver, m, read_first=False)
    want = loaded_run(solver, m, read_first=True)
    for i, (g, w) in enumerate(zip(got, want)):
        assert same_bits(g[0], w[0]), (i, g[0], w[0])
        assert g[1] == w[1], (i, g[1], w[1])
        assert same_bits(g[2], w[2]) and same_bits(g[3], w[3]), i
    # the loaded scores were consumed: the run differs from one that never loaded them
    assert not same_bits(got[0][0], loaded_run(solver, None, read_first=False)[0][0])
