"""Argument checks of the one-shot prediction path (api.predict / primalcr_predict), which shares its device checks and
id scans with primalcr_recommend, primalcr_similar and primalcr_rank_heldout."""
import numpy as np
import pytest

from primalcr_b200 import api


def factors(d1=4, d2=6, k=3):
    """Integer-valued factors: every product and sum is exact, so any summation order gives the same bits."""
    rng = np.random.default_rng(7)
    return rng.integers(-9, 10, (d1, k)).astype(np.float64), rng.integers(-9, 10, (d2, k)).astype(np.float64)


def raw_predict(U, V, users, items, out, device):
    return api.lib().primalcr_predict(U.ctypes.data, U.shape[0], V.ctypes.data, V.shape[0], U.shape[1],
                                      users.ctypes.data, items.ctypes.data, len(users), out.ctypes.data, device)


# ----------------------------------------------------------------------------- CPU
def test_predict_rejects_mismatched_factor_columns():
    U, _ = factors()
    V = np.ones((6, 2))
    with pytest.raises(api.PrimalCRError, match="same number of columns"):
        api.predict(U, V, [0, 1], [2, 3])


def test_predict_rejects_mismatched_id_lengths():
    U, V = factors()
    with pytest.raises(api.PrimalCRError, match="same length"):
        api.predict(U, V, [0, 1, 2], [2, 3])
    with pytest.raises(api.PrimalCRError, match="1-D"):
        api.predict(U, V, [[0, 1]], [[2, 3]])


def test_predict_without_gpu_fails_loudly(have_gpu):
    if have_gpu:
        pytest.skip("a GPU is present")
    U, V = factors()
    users = np.array([0, 3], np.int32); items = np.array([5, 0], np.int32); out = np.empty(2)
    assert raw_predict(U, V, users, items, out, 0) == -2
    assert "no CPU fallback" in api.lib().primalcr_last_error().decode()


# ----------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_predict_bad_device_ordinal_is_an_argument_error():
    U, V = factors()
    users = np.array([0, 3, 1, 3], np.int32); items = np.array([5, 0, 2, 2], np.int32); out = np.empty(4)
    assert raw_predict(U, V, users, items, out, 99) == -1
    assert "bad device ordinal" in api.lib().primalcr_last_error().decode()
    assert raw_predict(U, V, users, items, out, 0) == 0          # a valid call afterwards
    assert np.array_equal(out, np.einsum("ij,ij->i", U[users], V[items]))
