"""The xsim oracle (oracle/xsim.py) against an INDEPENDENT implementation: scikit-learn's brute-force cosine k-NN for the
neighbour search (its results on these seeded inputs are stored in tests/golden/xsim_sklearn_knn.pt, made by
tests/golden/make_xsim_sklearn_golden.py), and a literal dense evaluation of the LASER margin formula for the scoring.  The
reference itself has no xsim code (README.md:5 names the task only), so this is the strongest pin available offline; CPU only."""

import os

import numpy as np
import pytest
import torch

from oracle import xsim as ox

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "xsim_sklearn_knn.pt")
CASES = [(200, 300, 64, 4), (257, 129, 32, 5), (64, 64, 16, 1)]


def case_key(n, m, d, k):
    return f"n{n}_m{m}_d{d}_k{k}"


def _data(n, m, d, seed, noise=0.3):
    g = np.random.default_rng(seed)
    y = g.standard_normal((m, d)).astype(np.float32)
    x = (y[:n] if n <= m else g.standard_normal((n, d)).astype(np.float32)).copy()
    x += noise * g.standard_normal(x.shape).astype(np.float32)
    return x, y


@pytest.fixture(scope="module")
def sklearn_knn():
    return torch.load(GOLDEN, weights_only=True)


@pytest.mark.parametrize("n,m,d,k", CASES)
def test_oracle_knn_equals_sklearn_brute_force_cosine(sklearn_knn, n, m, d, k):
    x, y = _data(n, m, d, seed=n + m)
    val, idx = ox.knn(x, y, k)
    ref = sklearn_knn[case_key(n, m, d, k)]
    ind, dist = ref["indices"].numpy(), ref["distances"].numpy()
    assert ind.shape == (n, k)
    assert np.array_equal(idx, ind)
    np.testing.assert_allclose(val, 1.0 - dist, rtol=0, atol=1e-12)


@pytest.mark.parametrize("margin", ["ratio", "distance", "absolute"])
def test_oracle_margin_equals_the_dense_formula(margin):
    """LASER xsim: score(x_i, y_j) = margin(cos(x_i, y_j), (avg of x_i's k best cosines + avg of y_j's k best cosines) / 2),
    evaluated here for EVERY pair from the dense cosine matrix; the prediction is the best-scoring one of x_i's k nearest
    candidates."""
    n, k = 150, 4
    x, y = _data(n, n, 48, seed=5, noise=0.8)
    xn = x.astype(np.float64) / np.linalg.norm(x.astype(np.float64), axis=1, keepdims=True)
    yn = y.astype(np.float64) / np.linalg.norm(y.astype(np.float64), axis=1, keepdims=True)
    cos = xn @ yn.T
    avg_x = np.sort(cos, axis=1)[:, -k:].mean(axis=1)
    avg_y = np.sort(cos, axis=0)[-k:, :].mean(axis=0)
    denom = (avg_x[:, None] + avg_y[None, :]) / 2.0
    dense = {"ratio": cos / denom, "distance": cos - denom, "absolute": cos}[margin]
    cand = np.argsort(-cos, axis=1, kind="stable")[:, :k]
    want = cand[np.arange(n), np.argmax(np.take_along_axis(dense, cand, axis=1), axis=1)]
    err, total, pred = ox.xsim(x, y, margin=margin, k=k)
    assert total == n and np.array_equal(pred, want)
    assert err == int((want != np.arange(n)).sum())
