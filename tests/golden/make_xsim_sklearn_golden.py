"""Generate tests/golden/xsim_sklearn_knn.pt: scikit-learn's brute-force cosine k-NN (an INDEPENDENT implementation of the
neighbour search `oracle/xsim.py::knn` restates) on the seeded inputs of tests/test_oracle_xsim.py, one entry per case:
neighbour indices and cosine distances, both float64 maths.

    python tests/golden/make_xsim_sklearn_golden.py"""

import os
import sys

import numpy as np
import torch
from sklearn.neighbors import NearestNeighbors

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from tests.test_oracle_xsim import CASES, _data, case_key  # noqa: E402


def main() -> None:
    out = {}
    for n, m, d, k in CASES:
        x, y = _data(n, m, d, seed=n + m)
        nn = NearestNeighbors(n_neighbors=k, metric="cosine", algorithm="brute").fit(y.astype(np.float64))
        dist, ind = nn.kneighbors(x.astype(np.float64))
        out[case_key(n, m, d, k)] = {"indices": torch.from_numpy(ind), "distances": torch.from_numpy(dist)}
    torch.save(out, os.path.join(HERE, "xsim_sklearn_knn.pt"))
    print("wrote xsim_sklearn_knn.pt", list(out))


if __name__ == "__main__":
    main()
