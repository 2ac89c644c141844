"""The K-medoids oracle (oracle/select_oracle.py) against the goldens produced by the reference's own
KMedoids class (tests/golden/make_select_golden.py -> select_golden.npz)."""
import os
import warnings

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import select_oracle as so


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(GOLDEN, "select_golden.npz")))


def _kwargs(g, name):
    return dict(eval(str(g[name + "_kwargs"])))


def test_oracle_reproduces_the_reference_class(golden):
    for name in golden["names"]:
        D = golden[name + "_D"]
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            labels, medoids, n_iter = so.kmedoids_fit(D, **_kwargs(golden, name))
        assert np.array_equal(labels, golden[name + "_labels"]), name
        assert n_iter == int(golden[name + "_n_iter"]), name
        # duplicated points have identical rows: compare the medoids' rows, not their indices
        assert np.array_equal(D[medoids], D[golden[name + "_medoids"]]), name
        assert sum("is empty" in str(w.message) for w in caught) == int(golden[name + "_empty_warnings"]), name


def test_knn_oracle_is_sklearns_graph():
    rng = np.random.default_rng(3)
    P = rng.random((40, 5))
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    idx, dist = so.knn_graph(D, 7)
    assert idx.shape == (40, 7) and (idx != np.arange(40)[:, None]).all()
    assert np.all(np.diff(dist, axis=1) >= 0)
    assert np.array_equal(dist, np.take_along_axis(D, idx, axis=1))
