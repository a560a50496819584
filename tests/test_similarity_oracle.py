"""The similarity reference ko_similarity (tests/similarity_oracle.c) that the nearest_neighbors tests compare against,
pinned two ways without a GPU: bit for bit against a numpy float32 restatement of the canonical sequence, and against
float64 within the error bound of the blocked sum."""
import numpy as np
import pytest

import similarity_oracle as S

METRICS = ("dot", "cosine", "l2", "l1")
U = 2.0 ** -24


def terms(metric, Q, X):
    q, x = Q[:, None, :], X[None, :, :]
    if metric == "l2":
        t = q - x
        return t * t
    if metric == "l1":
        return np.abs(q - x)
    return q * x


def acc32(T):
    """Blocks of 32 along the last axis, each summed in index order from +0.0f; block sums added in index order."""
    a = np.zeros(T.shape[:-1], dtype=np.float32)
    for k0 in range(0, T.shape[-1], 32):
        part = np.zeros(T.shape[:-1], dtype=np.float32)
        for k in range(k0, min(k0 + 32, T.shape[-1])):
            part = part + T[..., k]
        a = a + part
    return a


def numpy_similarity(X, Q, metric):
    a = acc32(terms("dot" if metric == "cosine" else metric, Q, X))
    if metric == "cosine":
        qn = np.sqrt(acc32(Q * Q))
        xn = np.sqrt(acc32(X * X))
        return a / (qn[:, None] * xn[None, :])
    if metric == "l2":
        return -np.sqrt(a)
    return -a if metric == "l1" else a


def same_bits(a, b):
    a, b = a.copy(), b.copy()
    assert np.array_equal(np.isnan(a), np.isnan(b))
    a[np.isnan(a)] = 0.0
    b[np.isnan(b)] = 0.0
    return np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("width", [1, 23, 32, 37, 100])
@pytest.mark.parametrize("metric", METRICS)
def test_oracle_matches_numpy_float32_bit_for_bit(metric, width):
    rng = np.random.RandomState(width)
    X = rng.standard_normal((41, width)).astype(np.float32)
    X[3] = 0.0                                          # cosine: 0/0 = NaN
    X[4] = X[5]                                         # duplicate rows
    Q = np.concatenate([X[:5], rng.standard_normal((6, width)).astype(np.float32) * 7]).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        want = numpy_similarity(X, Q, metric)
    got = S.similarity(X, Q, metric)
    assert got.shape == (Q.shape[0], X.shape[0]) and got.dtype == np.float32
    assert same_bits(got, want), metric
    if metric == "cosine":
        assert np.isnan(got[:, 3]).all() and np.isnan(got[3]).all()


@pytest.mark.parametrize("width", [5, 64, 1000, 2000])
@pytest.mark.parametrize("metric", METRICS)
def test_oracle_within_the_blocked_sum_bound_of_float64(metric, width):
    rng = np.random.RandomState(100 + width)
    X = (rng.standard_normal((50, width)) * rng.uniform(0.01, 3.0, size=(50, 1))).astype(np.float32)
    Q = (rng.standard_normal((7, width)) * 2).astype(np.float32)
    got = S.similarity(X, Q, metric).astype(np.float64)
    X64, Q64 = X.astype(np.float64), Q.astype(np.float64)
    gamma = (32 + width / 32) * U                       # relative bound of the blocked sum (Higham, for sums of depth n)
    T = terms("dot" if metric == "cosine" else metric, Q64, X64)
    exact, bound = T.sum(-1), gamma * np.abs(T).sum(-1)
    if metric == "dot":
        assert (np.abs(got - exact) <= bound).all()
    elif metric == "l1":
        assert (np.abs(-got - exact) <= bound).all()
    elif metric == "l2":                                # s = -fl(sqrt(a)): s^2 = a (1 + e)^2, |e| <= 2^-24
        assert (np.abs(got * got - exact) <= bound + 2.01 * U * (exact + bound)).all()
    else:
        qn = np.sqrt((Q64 * Q64).sum(-1))[:, None]
        xn = np.sqrt((X64 * X64).sum(-1))[None, :]
        cos = exact / (qn * xn)
        # the dot product's absolute error, and the relative errors of the two norms (gamma / 2 + one sqrt rounding
        # each), the product and the quotient
        assert (np.abs(got - cos) <= 1.001 * (bound / (qn * xn) + np.abs(cos) * (gamma + 4 * U))).all()


def test_topk_helper_orders_ties_by_id_and_nan_last():
    s = np.array([[1.0, np.nan, 2.0, 1.0, -0.0, 0.0, -np.inf]], dtype=np.float32)
    ids, scores = S.topk(s, 9)
    assert ids.tolist() == [[2, 0, 3, 4, 5, 6, 1, -1, -1]]
    assert np.isneginf(scores[0, 7:]).all()
    ids, _ = S.topk(s, 3, self_ids=np.array([2]))
    assert ids.tolist() == [[0, 3, 4]]
