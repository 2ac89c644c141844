"""HDBSCAN without a GPU: the numpy oracle (oracle/hdbscan_oracle.py) against scikit-learn's HDBSCAN, and the
library's host stage (po_hdbscan_tree: single-linkage tree, condensed tree, stability, excess of mass,
labels, probabilities) against the oracle, bit for bit."""
import functools

import numpy as np
import pytest
from sklearn.cluster import HDBSCAN as SkHDBSCAN

from oracle import hdbscan_oracle as ho
from oracle import phylo_oracle as po
from phyloligo_b200 import phyloselect, synth


@functools.lru_cache(maxsize=None)
def blobs(n, seed, dim=4, centres=6, spread=6.0):
    rng = np.random.default_rng(seed)
    c = rng.normal(0, spread, size=(centres, dim))
    P = c[rng.integers(0, centres, n)] + rng.normal(0, 1, size=(n, dim))
    D = np.sqrt(((P[:, None, :] - P[None, :, :]) ** 2).sum(-1))
    D.flags.writeable = False  # shared between tests
    return D


@functools.lru_cache(maxsize=None)
def jsd_matrix(n, seed, mean_len=3000):
    seqs = synth.make_sequences(n, mean_len, seed=seed)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs])
    D = po.pairwise_np(X, "JSD").astype(np.float32)
    D.flags.writeable = False  # shared between tests
    return D


def tied_endpoints(u, v, w):
    """Endpoints of MST edges whose weight another MST edge shares."""
    vals, counts = np.unique(w, return_counts=True)
    shared = np.isin(w, vals[counts > 1])
    return set(u[shared].tolist()) | set(v[shared].tolist())


def assert_same_clustering(ours, probs, theirs, their_probs, exempt=frozenset()):
    """Equal labels up to the numbering of the clusters (noise is -1 on both sides) and probabilities within
    1e-12, except at the exempt points."""
    keep = np.array([i not in exempt for i in range(len(ours))])
    mapping = {}
    for a, b in zip(ours[keep].tolist(), theirs[keep].tolist()):
        assert mapping.setdefault(a, b) == b, "cluster %d maps to %d and %d" % (a, mapping[a], b)
    assert mapping.get(-1, -1) == -1
    assert len(set(mapping.values())) == len(mapping), "two clusters map to one"
    assert np.array_equal(np.vectorize(mapping.get)(ours[keep]), theirs[keep])
    assert np.abs(probs[keep] - their_probs[keep]).max(initial=0.0) <= 1e-12


CASES = [("blobs", 50, 1, 5, None), ("blobs", 300, 2, 5, 1), ("blobs", 1000, 3, 15, 3), ("blobs", 3000, 4, 40, None),
         ("blobs", 700, 5, 5, None), ("jsd", 400, 11, 5, None), ("jsd", 1500, 7, 5, 1), ("jsd", 1500, 7, 15, 3),
         ("jsd", 800, 12, 40, None), ("blobs", 1000, 3, 5, 1), ("blobs", 2000, 11, 5, 1)]
# the cases whose MST weights are all distinct (the MST is unique; no point is exempt from the comparison)
DISTINCT = {("blobs", 300, 2, 5, 1), ("jsd", 1500, 7, 5, 1), ("blobs", 1000, 3, 5, 1), ("blobs", 2000, 11, 5, 1)}


@pytest.mark.parametrize("kind,n,seed,mcs,ms", CASES)
def test_oracle_matches_scikit_learn(kind, n, seed, mcs, ms):
    D = blobs(n, seed) if kind == "blobs" else jsd_matrix(n, seed)
    res = ho.hdbscan(D, mcs, ms)
    msc = ho.clamp_min_samples(n, mcs, ms)
    # scikit-learn's min_samples counts the point itself
    sk = SkHDBSCAN(min_cluster_size=mcs, min_samples=msc + 1, metric="precomputed", copy=True).fit(D.astype(np.float64))
    u, v, w = res["mst"]
    assert len(u) == n - 1 and (u < v).all()
    distinct = len(np.unique(w)) == len(w)
    assert distinct == ((kind, n, seed, mcs, ms) in DISTINCT)
    exempt = frozenset() if distinct else tied_endpoints(u, v, w)
    assert_same_clustering(res["labels"], res["probabilities"], sk.labels_, sk.probabilities_, exempt)


def test_kruskal_and_streaming_prim_agree():
    for D, ms in [(blobs(400, 8), 5), (jsd_matrix(300, 9), 3), (np.round(blobs(300, 10), 0), 4)]:
        core = ho.core_distances(D, ms)
        a, b = ho.mst_kruskal(D, core), ho.mst_prim_streaming(D, core)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


def host_stage(D, mcs, ms=None, seed=0):
    """The oracle's result and the library's host stage fed the oracle's MST, shuffled and flipped."""
    n = D.shape[0]
    res = ho.hdbscan(D, mcs, ms)
    u, v, w = res["mst"]
    rng = np.random.default_rng(seed)
    perm = rng.permutation(n - 1)
    flip = rng.random(n - 1) < 0.5
    uu, vv = np.where(flip, v, u)[perm], np.where(flip, u, v)[perm]
    ww = w[perm].astype(np.float64)
    before = (uu.copy(), vv.copy(), ww.copy())
    out = phyloselect.hdbscan_tree(uu, vv, ww, n, mcs)
    assert all(np.array_equal(a, b) for a, b in zip((uu, vv, ww), before))  # the inputs are left alone
    return res, out


def assert_host_equals_oracle(res, out, n, mcs):
    labels, probs, ct, slt, mst = out
    assert np.array_equal(labels, res["labels"])
    assert np.array_equal(probs, res["probabilities"])
    oct_ = res["condensed_tree"]
    assert len(ct) == len(oct_)
    for f in ("parent", "child", "lambda_val", "child_size"):
        assert np.array_equal(ct[f], oct_[f]), f
    u, v, w = res["mst"]
    assert np.array_equal(mst, np.column_stack([u, v, w]).astype(np.float64))  # tie-rule order, u < v
    left, right, dist, size = ho.single_linkage(u, v, w, n)
    assert np.array_equal(slt, np.column_stack([left, right, dist, size]).astype(np.float64))


@pytest.mark.parametrize("kind,n,seed,mcs,ms", CASES[:5] + CASES[6:8])
def test_host_stage_equals_the_oracle(kind, n, seed, mcs, ms):
    D = blobs(n, seed) if kind == "blobs" else jsd_matrix(n, seed)
    res, out = host_stage(D, mcs, ms, seed)
    assert_host_equals_oracle(res, out, n, mcs)


def test_host_stage_orders_tied_edges_by_the_tie_rule():
    D = np.round(blobs(200, 3), 0)  # a handful of distinct weights
    res, out = host_stage(D, 5)
    assert len(np.unique(res["mst"][2])) < 20
    assert_host_equals_oracle(res, out, 200, 5)


def test_duplicate_contigs_give_infinite_lambda():
    P = np.random.default_rng(4).normal(0, 1, size=(60, 3))
    P = np.vstack([P, P[:20], P[:20]])  # every one of the first 20 points three times
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    res, out = host_stage(D, 3, 1)
    assert np.isinf(res["condensed_tree"]["lambda_val"]).any()
    assert_host_equals_oracle(res, out, len(P), 3)


def test_all_noise():
    D = blobs(40, 6, centres=40, spread=50.0)  # isolated points: no split has two sides of min_cluster_size
    res, out = host_stage(D, 8)
    assert (res["labels"] == -1).all()
    assert_host_equals_oracle(res, out, 40, 8)


def test_a_single_dense_blob_is_all_noise():
    D = blobs(150, 7, centres=1)
    res, out = host_stage(D, 80)
    assert (res["condensed_tree"]["parent"] == 150).all()  # the root only
    assert (res["labels"] == -1).all() and (res["probabilities"] == 0).all()
    assert_host_equals_oracle(res, out, 150, 80)


@pytest.mark.parametrize("n", [2, 3])
def test_tiny_inputs(n):
    D = blobs(n, n)
    res, out = host_stage(D, 2)
    assert_host_equals_oracle(res, out, n, 2)
    sk = SkHDBSCAN(min_cluster_size=2, min_samples=n, metric="precomputed", copy=True).fit(D)
    assert_same_clustering(res["labels"], res["probabilities"], sk.labels_, sk.probabilities_)


def test_min_samples_at_least_n_minus_1():
    D = blobs(30, 9)
    for ms in (29, 40):
        res, out = host_stage(D, 5, ms)
        assert_host_equals_oracle(res, out, 30, 5)
        assert (res["core"] == D.max(axis=1)).all()  # the largest entry of every row


def test_host_stage_refuses_a_cycle():
    with pytest.raises(phyloselect.PhyloligoError, match="cycle"):
        phyloselect.hdbscan_tree(np.array([0, 1, 0]), np.array([1, 0, 2]), np.array([1.0, 2.0, 3.0]), 4, 2)


@pytest.mark.parametrize("kwargs,what", [
    ({"min_cluster_size": 1}, "min_cluster_size=1"), ({"min_cluster_size": 0}, "min_cluster_size=0"),
    ({"min_samples": 0}, "min_samples=0"), ({"alpha": 2.0}, "alpha"), ({"cluster_selection_method": "leaf"}, "cluster_selection_method"),
    ({"allow_single_cluster": True}, "allow_single_cluster"), ({"cluster_selection_epsilon": 0.5}, "cluster_selection_epsilon"),
    ({"metric": "cosine"}, "cosine"), ({"colour": 3}, "colour")])
def test_constructor_refuses(kwargs, what):
    with pytest.raises(ValueError, match=what):
        phyloselect.HDBSCAN(**kwargs)


def test_constructor_accepts_contrib_defaults():
    h = phyloselect.HDBSCAN(min_cluster_size=7, min_samples=2, alpha=1.0, cluster_selection_method="eom",
                            allow_single_cluster=False, cluster_selection_epsilon=0.0)
    assert (h.min_cluster_size, h.min_samples, h.metric) == (7, 2, "precomputed")
