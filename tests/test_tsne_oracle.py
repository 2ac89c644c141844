"""t-SNE without a GPU: the numpy oracle (oracle/tsne_oracle.py) against scikit-learn's TSNE(method="barnes_hut",
angle=0.0) -- its joint probabilities, its gradient and KL, and a whole fit -- and the argument refusals of
phyloselect.TSNE, which happen before any device work."""
import numpy as np
import pytest
from sklearn.manifold import TSNE as SkTSNE
from sklearn.manifold import _t_sne, trustworthiness
from sklearn.neighbors import NearestNeighbors

from oracle import tsne_oracle as to
from phyloligo_b200 import phyloselect
from test_hdbscan_oracle import blobs, jsd_matrix


def matrix(kind, n, seed):
    return blobs(n, seed) if kind == "blobs" else jsd_matrix(n, seed)


def sklearn_P(D, perplexity):
    n = D.shape[0]
    k = min(n - 1, int(3.0 * perplexity + 1))
    G = NearestNeighbors(n_neighbors=k, metric="precomputed").fit(D).kneighbors_graph(mode="distance")
    G.data **= 2
    return _t_sne._joint_probabilities_nn(G, perplexity, 0).tocsr()


def sklearn_gradient(P, Y, exaggeration=1.0):
    n = Y.shape[0]
    Pe = P.copy()
    Pe.data = Pe.data * exaggeration
    err, g = _t_sne._kl_divergence_bh(np.asarray(Y, np.float32).ravel().copy(), Pe, 1, n, 2, angle=0.0, compute_error=True,
                                      num_threads=1)
    return g.reshape(n, 2), err


CASES = [("blobs", 400, 1, 30.0), ("blobs", 300, 2, 100.0), ("jsd", 300, 3, 30.0), ("jsd", 250, 4, 5.0)]


@pytest.mark.parametrize("kind,n,seed,perplexity", CASES)
def test_joint_probabilities_equal_scikit_learn(kind, n, seed, perplexity):
    D = matrix(kind, n, seed)
    want = sklearn_P(D, perplexity)
    got = to.joint_probabilities(D, perplexity)
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.abs(got.data - want.data).max() <= 1e-12


@pytest.mark.parametrize("kind,n,seed,perplexity", CASES[:3])
@pytest.mark.parametrize("exaggeration", [1.0, 12.0])
def test_gradient_and_kl_equal_scikit_learn_exact_barnes_hut(kind, n, seed, perplexity, exaggeration):
    D = matrix(kind, n, seed)
    P = sklearn_P(D, perplexity)
    Y = np.random.default_rng(seed).normal(0, 3, size=(n, 2)).astype(np.float32)
    g_want, kl_want = sklearn_gradient(P, Y, exaggeration)
    g, kl = to.gradient(P, Y, exaggeration)
    assert np.abs(g - g_want).max() <= 1e-5 * np.abs(g_want).max()
    # scikit-learn accumulates the KL terms in a float32 variable: about 1e-5 of rounding at these sizes
    assert abs(kl - kl_want) <= 5e-5 * abs(kl_want)


@pytest.mark.parametrize("kind,n,seed", [("blobs", 500, 1), ("jsd", 400, 3)])
def test_full_fit_matches_scikit_learn(kind, n, seed):
    D = matrix(kind, n, seed)
    sk = SkTSNE(metric="precomputed", init="random", random_state=0, angle=0.0).fit(np.array(D))
    res = to.fit(D, random_state=0)
    assert res["learning_rate"] == sk.learning_rate_
    assert abs(res["kl_divergence"] - sk.kl_divergence_) <= 0.01 * sk.kl_divergence_
    t_sk = trustworthiness(D, sk.embedding_, n_neighbors=10, metric="precomputed")
    t_or = trustworthiness(D, res["embedding"], n_neighbors=10, metric="precomputed")
    assert abs(t_sk - t_or) <= 0.005


def test_random_init_is_scikit_learns_draw():
    # TSNE(init="random") draws 1e-4 * standard_normal((n, 2)).astype(float32) from check_random_state(seed)
    from sklearn.utils import check_random_state
    for seed in (0, 7):
        want = 1e-4 * check_random_state(seed).standard_normal(size=(50, 2)).astype(np.float32)
        assert np.array_equal(to.random_init(50, seed), want)
        assert np.array_equal(1e-4 * phyloselect._random_state(seed).standard_normal(size=(50, 2)).astype(np.float32), want)


@pytest.mark.parametrize("kwargs,message", [
    ({"method": "exact"}, "method='exact' is not supported"),
    ({"angle": 0.5}, "angle=0.5 is not supported"),
    ({"verbose": 1}, "verbose=1 is not supported"),
    ({"metric_params": {"p": 1}}, "metric_params=.* is not supported"),
    ({"n_jobs": 4}, "n_jobs=4 is not supported"),
    ({"n_components": 3}, "n_components=3 is not supported"),
    ({"init": "pca"}, 'init="pca" cannot be used with metric="precomputed"'),
    ({"init": "spectral"}, "init must be 'random' or an"),
    ({"perplexity": 0.0}, "perplexity must be positive"),
    ({"early_exaggeration": 0.5}, "early_exaggeration must be at least 1"),
    ({"learning_rate": -1.0}, "learning_rate must be 'auto' or positive"),
    ({"max_iter": 100}, "max_iter must be an integer of at least 250"),
    ({"metric": "cosine"}, "metric needs to be 'precomputed' or one of"),
])
def test_refused_arguments(kwargs, message):
    with pytest.raises(ValueError, match=message):
        phyloselect.TSNE(**kwargs)


def test_accepted_arguments():
    t = phyloselect.TSNE(method="barnes_hut", angle=0.0, verbose=0, metric_params=None, n_jobs=None, learning_rate=200.0,
                         init=np.zeros((5, 2)), metric="JSD", perplexity=5)
    assert t.perplexity == 5 and t.metric == "JSD"
