#!/usr/bin/env python3
"""The front half of phyloselect.py on B200 (SURVEY.md 8f rank 4): K-medoids, HDBSCAN and the t-SNE projection
of the contig distance matrix, and phyloselect.R's hierarchical tree, computed on the device while the matrix is resident -- straight after the
distance stage if wanted, without the round trip through a 40 GB file and 800 GB of host RAM the reference's documentation asks for.

Mirrors reference phylopackage/bin/phyloselect.py: ``KMedoids`` (:37-309; same constructor
arguments and fitted attributes), ``clusterize`` (:573-590), ``find_clusters`` (:403-428), the
matrix readers of ``main`` (:597-622), ``write_fastafile`` (:547-571) and the
``data_cluster_indexes.dat`` writer (:742-751).  ``HDBSCAN`` computes what the reference gets from
the third-party hdbscan.HDBSCAN(metric="precomputed") with its default arguments (core distances,
mutual-reachability MST, condensed tree, excess-of-mass selection), with MST ties broken by vertex
index.  ``TSNE`` computes what the reference gets from sklearn.manifold.TSNE(metric="precomputed") (:381-398)
with angle=0.0, i.e. the exact gradient; ``--tsne-out`` writes its embedding.  ``linkage`` / ``HClust`` build the
tree bin/phyloselect.R:22-35 builds with hclust, as scipy.cluster.hierarchy.linkage computes it; ``-m hclust`` cuts
it and ``--tree-out`` writes it in Newick format.  ``nj`` builds the neighbour-joining trees the same script offers
(ape's nj and bionj, in the operation order DESIGN.md section 4.11 fixes); ``--tree-method nj|bionj`` makes ``--tree-out`` write one.
Plotting and the interactive loop are out of scope.

There is no CPU fallback: the sums, assignments, selections, the MST, the t-SNE gradient, the linkage loop and the
neighbour joins run in libphyloligo_b200.so.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import sys
import warnings

import numpy as np
import torch

from . import _lib, engine, io_formats, panels
from ._lib import PhyloligoError, PO_F32, PO_F64


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dt(D):
    if D.dtype == torch.float32:
        return PO_F32
    if D.dtype == torch.float64:
        return PO_F64
    raise PhyloligoError("the distance matrix must be float32 or float64")


def as_device_matrix(D):
    """A 2-D float32 / float64 device tensor with contiguous rows from an ndarray / memmap / tensor."""
    device = engine.require_cuda()
    if isinstance(D, torch.Tensor):
        t = D.to(device)
    else:
        a = np.asarray(D)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        t = torch.from_numpy(np.ascontiguousarray(a)).to(device)
    if t.dim() != 2 or t.shape[0] != t.shape[1]:
        raise PhyloligoError("a square distance matrix is expected, got shape %s" % (tuple(t.shape),))
    if t.stride(1) != 1:
        t = t.contiguous()
    _dt(t)
    return t


def _source(X, metric):
    """The row-panel source (panels.py) a fit reads: X itself when it is one; for "precomputed" the matrix X
    (resident, or read in panels from a matrix file that does not fit on the device); otherwise the matrix of the
    profiles X for `metric`, resident when it fits in device memory and recomputed panel by panel when not."""
    if isinstance(X, panels.SOURCES):
        return X
    if metric == "precomputed":
        return panels.as_source(X)
    return panels.profile_source(X, metric)


def row_sums(D, rows=None, labels=None, row_labels=None):
    """float64 sums of rows of the device matrix D (po_matrix_rowsums): all columns, or only the columns j
    with labels[j] == row_labels[i]."""
    lib = _lib.load()
    n_cols = int(D.shape[1])
    n_rows = int(rows.shape[0]) if rows is not None else int(D.shape[0])
    out = torch.empty(n_rows, dtype=torch.float64, device=D.device)
    rc = lib.po_matrix_rowsums(_ptr(D), int(D.stride(0)), _dt(D), _ptr(rows), n_rows, n_cols, _ptr(labels), _ptr(row_labels),
                               _ptr(out), _stream())
    _lib.check(rc, "po_matrix_rowsums")
    return out


def assign_to_medoids(D, medoids):
    """labels[j] = argmin_c D[medoids[c], j] (po_matrix_argmin_rows), int32."""
    lib = _lib.load()
    n = int(D.shape[1])
    out = torch.empty(n, dtype=torch.int32, device=D.device)
    rc = lib.po_matrix_argmin_rows(_ptr(D), int(D.stride(0)), _dt(D), _ptr(medoids), int(medoids.shape[0]), n, _ptr(out), _stream())
    _lib.check(rc, "po_matrix_argmin_rows")
    return out


def cluster_argmin(cost, labels, k):
    """(best_idx int64[k], best_cost float64[k], count int64[k]) per cluster (po_cluster_argmin)."""
    lib = _lib.load()
    dev = cost.device
    work = torch.empty(2 * k, dtype=torch.int64, device=dev)
    best_idx = torch.empty(k, dtype=torch.int64, device=dev)
    best_cost = torch.empty(k, dtype=torch.float64, device=dev)
    count = torch.empty(k, dtype=torch.int64, device=dev)
    rc = lib.po_cluster_argmin(_ptr(cost), _ptr(labels), int(cost.shape[0]), int(k), _ptr(work), _ptr(best_idx), _ptr(best_cost),
                               _ptr(count), _stream())
    _lib.check(rc, "po_cluster_argmin")
    return best_idx, best_cost, count


def _knn_rows(P, self0, k, idx, dist):
    """po_matrix_knn of the rows of the device view P (row i is matrix row self0 + i) into idx / dist."""
    rc = _lib.load().po_matrix_knn(_ptr(P), int(P.stride(0)), _dt(P), int(P.shape[0]), int(P.shape[1]), int(self0), int(k),
                                   _ptr(idx), _ptr(dist), _stream())
    _lib.check(rc, "po_matrix_knn")


def knn_graph(D, k, row0=0, as_sparse=False):
    """The k nearest neighbours of every row of the device matrix D (a block row when row0 > 0: row i is
    profile row0 + i and that column is excluded), ascending, ties by column (po_matrix_knn).  D may also be a
    row-panel source (panels.py): one pass over its panels.
    Returns (indices int32 [n, k], distances float32 [n, k]) device tensors, or with `as_sparse` the
    scipy CSR matrix that sklearn's TSNE(metric="precomputed") / kneighbors_graph(mode="distance") use."""
    if isinstance(D, panels.SOURCES):
        parts = ((r0, r1, P) for r0, r1, P in D.panels())
        n_rows, n_cols, dev = D.n, D.n, D.device
    else:
        D = D if isinstance(D, torch.Tensor) and D.is_cuda else as_device_matrix(D)
        n_rows, n_cols, dev = int(D.shape[0]), int(D.shape[1]), D.device
        parts = [(0, n_rows, D)]
        row0 = int(row0)
    idx = torch.empty((n_rows, k), dtype=torch.int32, device=dev)
    dist = torch.empty((n_rows, k), dtype=torch.float32, device=dev)
    for r0, r1, P in parts:
        _knn_rows(P, r0 if isinstance(D, panels.SOURCES) else row0, k, idx[r0:r1], dist[r0:r1])
    if not as_sparse:
        return idx, dist
    from scipy.sparse import csr_matrix
    indptr = np.arange(0, n_rows * k + 1, k)
    return csr_matrix((dist.cpu().numpy().ravel().astype(np.float64), idx.cpu().numpy().ravel(), indptr), shape=(n_rows, n_cols))


class KMedoids:
    """k-medoids (PAM) on the device.  Same parameters and fitted attributes as the reference class
    (bin/phyloselect.py:37-309): ``labels_``, ``cluster_centers_`` (the medoids' rows of X), ``n_iter_``;
    ``medoid_indices_`` in addition.  ``distance_metric`` is "precomputed" (X is the N x N matrix: ndarray,
    memmap or a device tensor, which is used in place) or one of the package's metrics
    (Eucl, JSD, KT, BC, SC: X is the N x D profile matrix and the distances never leave the device)."""

    CLUSTERING_METHODS = ["pam"]
    INIT_METHODS = ["random", "heuristic"]

    def __init__(self, n_clusters=8, distance_metric="precomputed", clustering_method="pam", init="heuristic", max_iter=300,
                 random_state=None):
        self.n_clusters = n_clusters
        self.distance_metric = distance_metric
        self.init = init
        self.max_iter = max_iter
        self.clustering_method = clustering_method
        self.random_state = random_state

    def _check_init_args(self):
        if self.n_clusters is None or not isinstance(self.n_clusters, int) or self.n_clusters <= 0:
            raise ValueError("n_clusters has to be nonnegative integer")
        if self.distance_metric != "precomputed" and self.distance_metric not in _lib.METRICS:
            raise ValueError("distance_metric needs to be 'precomputed' or one of {}. Instead, '{}' was given.".format(
                sorted(_lib.METRICS), self.distance_metric))
        if self.clustering_method not in self.CLUSTERING_METHODS:
            raise ValueError("clustering must be one of the following: {}".format(self.CLUSTERING_METHODS))
        if self.init not in self.INIT_METHODS:
            raise ValueError("init needs to be one of the following: {}".format(self.INIT_METHODS))

    def fit(self, X, y=None):
        self._check_init_args()
        src = _source(X, self.distance_metric)
        n, k = src.n, self.n_clusters
        if k > n:
            raise ValueError("The number of medoids ({}) must be larger than the number of samples ({})".format(k, n))
        dev = src.device
        # initial medoids (:291-309)
        if self.init == "random":
            rs = self.random_state if isinstance(self.random_state, np.random.RandomState) else np.random.RandomState(self.random_state)
            medoids = torch.from_numpy(np.asarray(rs.permutation(n)[:k], dtype=np.int64)).to(dev)
        else:
            # np.argsort's order: NaN sums last whatever their sign (torch's device sort puts a negative NaN first)
            sums = torch.cat([row_sums(P) for _, _, P in src.panels()])
            nan = torch.isnan(sums)
            medoids = torch.argsort(torch.where(nan, torch.inf, sums), stable=True)
            medoids = medoids[torch.argsort(nan[medoids].to(torch.int8), stable=True)][:k].contiguous()
        cluster_ids = torch.arange(k, dtype=torch.int32, device=dev)
        old = None
        labels = None
        self.n_iter_ = 0
        while (old is None or not torch.equal(old, medoids)) and self.n_iter_ < self.max_iter:
            self.n_iter_ += 1
            old = medoids.clone()
            M = src.rows(medoids)                                                    # the medoids' rows, k x n
            labels = assign_to_medoids(M, cluster_ids.to(torch.int64))               # :187-195
            # every point's cost inside its own cluster
            cost = torch.cat([row_sums(P, labels=labels, row_labels=labels[r0:r1]) for r0, r1, P in src.panels()])
            curr = row_sums(M, labels=labels, row_labels=cluster_ids)               # the current medoids' costs (:207-211)
            best_idx, best_cost, count = cluster_argmin(cost, labels, k)             # :213-227
            empty = torch.nonzero(count == 0).flatten().tolist()
            for c in empty:
                warnings.warn("Cluster {} is empty!".format(c))
            better = (count > 0) & (best_cost < curr)                                # :229-240
            medoids = torch.where(better, best_idx, medoids)
        self.medoid_indices_ = medoids.cpu().numpy()
        self.labels_ = labels.cpu().numpy().astype(np.int64) if labels is not None else np.zeros(n, dtype=np.int64)
        if isinstance(X, panels.SOURCES):
            self.cluster_centers_ = X.rows(medoids).cpu().numpy()
        elif isinstance(X, torch.Tensor):
            self.cluster_centers_ = X[medoids.to(X.device)].cpu().numpy()
        else:
            self.cluster_centers_ = np.asarray(X).take(self.medoid_indices_, axis=0)
        return self


def check_matrix(D, row0=None, cols=None):
    """Refuse (PhyloligoError) a device matrix that is not square, not bitwise symmetric or holds a NaN or an
    infinite entry; the message names the first offending entry (po_hdbscan_check).  With row0, D is the row
    panel [row0, row0 + rows) of a square matrix of D.shape[1] rows, and `cols` its column strip (the
    transposed entries), or None for a source symmetric by construction (only the diagonal square is tested
    for symmetry); checked panel by panel in row order, the first failure names the entry the whole-matrix
    check names."""
    lib = _lib.load()
    work = torch.empty(1, dtype=torch.int64, device=D.device)
    if row0 is None:
        r0, cptr, cld = 0, None, 0
    else:
        r0, cptr, cld = int(row0), _ptr(cols), (int(cols.stride(0)) if cols is not None else max(1, int(D.shape[0])))
    rc = lib.po_hdbscan_check(_ptr(D), int(D.stride(0)), _dt(D), int(D.shape[0]), int(D.shape[1]), r0, cptr, cld, _ptr(work),
                              _stream())
    _lib.check(rc, "po_hdbscan_check")


def kth_smallest(D, k):
    """The k-th smallest entry (1-based, the diagonal counted) of every row of the device matrix D, bit for bit
    in D's dtype (po_matrix_kth)."""
    lib = _lib.load()
    out = torch.empty(int(D.shape[0]), dtype=D.dtype, device=D.device)
    rc = lib.po_matrix_kth(_ptr(D), int(D.stride(0)), _dt(D), int(D.shape[0]), int(D.shape[1]), int(k), _ptr(out), _stream())
    _lib.check(rc, "po_matrix_kth")
    return out


def mutual_reachability_mst(D, core, on_round=None):
    """The minimum spanning tree of mr(i, j) = max(core[i], core[j], D[i, j]) by Boruvka rounds on the device,
    edges compared by (mr, min(i, j), max(i, j)): every round scans the rows (po_hdbscan_mst_scan, one call per
    panel when D is a row-panel source) and then merges (po_hdbscan_mst_merge).  D must be bitwise symmetric
    (check_matrix).  Returns device tensors (u int64, v int64, w in D's dtype), n - 1 edges in no particular
    order.  `on_round(components)` is called after every round."""
    lib = _lib.load()
    src = D if isinstance(D, panels.SOURCES) else panels.ResidentSource(D)
    n, dev, dt = src.n, src.device, _dt(torch.empty(0, dtype=src.dtype))
    work = torch.empty(int(lib.po_hdbscan_mst_workspace(n)), dtype=torch.uint8, device=dev)
    u = torch.empty(max(n - 1, 1), dtype=torch.int64, device=dev)
    v = torch.empty_like(u)
    w = torch.empty(max(n - 1, 1), dtype=src.dtype, device=dev)
    _lib.check(lib.po_hdbscan_mst_init(n, _ptr(work), _stream()), "po_hdbscan_mst_init")
    comps = C.c_int64(n)
    while comps.value > 1:
        for r0, r1, P in src.panels():
            rc = lib.po_hdbscan_mst_scan(_ptr(P), int(P.stride(0)), dt, r0, r1 - r0, n, _ptr(core), _ptr(work), _stream())
            _lib.check(rc, "po_hdbscan_mst_scan")
        rc = lib.po_hdbscan_mst_merge(n, dt, _ptr(core), _ptr(work), _ptr(u), _ptr(v), _ptr(w), C.byref(comps), _stream())
        _lib.check(rc, "po_hdbscan_mst_merge")
        if on_round is not None:
            on_round(comps.value)
    return u[:n - 1], v[:n - 1], w[:n - 1]


CONDENSED_DTYPE = np.dtype([("parent", np.int64), ("child", np.int64), ("lambda_val", np.float64), ("child_size", np.int64)])


def hdbscan_tree(u, v, w, n, min_cluster_size):
    """Host stage (po_hdbscan_tree) from the n - 1 MST edges, in any order and orientation.  Returns (labels
    int64, probabilities float64, condensed tree, single-linkage tree n - 1 x 4, MST n - 1 x 3 of (i, j, w)
    with i < j in tie-rule order).  The inputs are not modified."""
    lib = _lib.load()
    u = np.array(u, dtype=np.int64)  # copies: the library sorts them in place
    v = np.array(v, dtype=np.int64)
    w = np.array(w, dtype=np.float64)
    m = n - 1
    if not (u.shape == v.shape == w.shape == (m,)):
        raise PhyloligoError("hdbscan_tree: %d points need %d edges" % (n, m))
    sl = [np.empty(m, np.int64), np.empty(m, np.int64), np.empty(m, np.float64), np.empty(m, np.int64)]
    cols = [np.empty(2 * n, np.int64), np.empty(2 * n, np.int64), np.empty(2 * n, np.float64), np.empty(2 * n, np.int64)]
    rows = np.zeros(1, np.int64)
    labels = np.empty(n, np.int64)
    probs = np.empty(n, np.float64)
    args = [u, v, w] + sl + cols + [rows, labels, probs]
    rc = lib.po_hdbscan_tree(n, int(min_cluster_size), *[C.c_void_p(a.ctypes.data) for a in args])
    _lib.check(rc, "po_hdbscan_tree")
    r = int(rows[0])
    ct = np.empty(r, dtype=CONDENSED_DTYPE)
    for name, col in zip(CONDENSED_DTYPE.names, cols):
        ct[name] = col[:r]
    slt = np.column_stack([sl[0].astype(np.float64), sl[1].astype(np.float64), sl[2], sl[3].astype(np.float64)])
    return labels, probs, ct, slt, np.column_stack([u.astype(np.float64), v.astype(np.float64), w])


class HDBSCAN:
    """HDBSCAN on the device.  Same parameters, defaults and fitted attributes as the hdbscan.HDBSCAN the
    reference calls (bin/phyloselect.py:403-428): ``labels_`` (-1 = noise), ``probabilities_``,
    ``minimum_spanning_tree_`` (n - 1 x 3 ndarray of (i, j, distance), i < j, sorted by the tie rule),
    ``condensed_tree_`` (structured ndarray: parent, child, lambda_val, child_size) and
    ``single_linkage_tree_`` (n - 1 x 4, scipy's linkage layout).  ``metric`` is "precomputed" (X is the
    N x N matrix: ndarray, memmap or a device tensor, which is used in place) or one of the package's metrics
    (X is the N x D profile matrix and the distances never leave the device).  Arguments of hdbscan.HDBSCAN
    other than min_cluster_size, min_samples and metric are accepted at their default values only.  MST
    edges of equal weight are ordered by (min(i, j), max(i, j)), which makes the result deterministic."""

    # hdbscan.HDBSCAN's other arguments and the only value accepted for each
    DEFAULTS = {"cluster_selection_epsilon": 0.0, "max_cluster_size": 0, "alpha": 1.0, "p": None, "algorithm": "best",
                "leaf_size": 40, "memory": None, "approx_min_span_tree": True, "gen_min_span_tree": False,
                "core_dist_n_jobs": 4, "cluster_selection_method": "eom", "allow_single_cluster": False,
                "prediction_data": False, "match_reference_implementation": False}

    def __init__(self, min_cluster_size=5, min_samples=None, metric="precomputed", **kwargs):
        for key, value in kwargs.items():
            if key not in self.DEFAULTS:
                raise ValueError("HDBSCAN has no argument {!r}".format(key))
            if value != self.DEFAULTS[key]:
                raise ValueError("{}={!r} is not supported; only the default {!r}".format(key, value, self.DEFAULTS[key]))
        if not isinstance(min_cluster_size, (int, np.integer)) or isinstance(min_cluster_size, bool) or (
                min_samples is not None and (not isinstance(min_samples, (int, np.integer)) or isinstance(min_samples, bool))):
            raise ValueError("Min samples and min cluster size must be integers!")
        if min_cluster_size <= 0 or (min_samples is not None and min_samples <= 0):
            raise ValueError("Min samples and Min cluster size must be positive integers (min_cluster_size={}, min_samples={})"
                             .format(min_cluster_size, min_samples))
        if min_cluster_size == 1:
            raise ValueError("Min cluster size must be greater than one (min_cluster_size=1)")
        if metric != "precomputed" and metric not in _lib.METRICS:
            raise ValueError("metric needs to be 'precomputed' or one of {}. Instead, '{}' was given.".format(sorted(_lib.METRICS), metric))
        self.min_cluster_size = int(min_cluster_size)
        self.min_samples = None if min_samples is None else int(min_samples)
        self.metric = metric

    def fit(self, X, y=None):
        src = _source(X, self.metric)
        n = src.n
        if n < 2:
            raise ValueError("HDBSCAN needs at least 2 samples, got {}".format(n))
        ms = min(self.min_cluster_size if self.min_samples is None else self.min_samples, n - 1)
        core = torch.empty(n, dtype=src.dtype, device=src.device)
        for r0, r1, P in src.panels():  # the check and the core distances: one pass
            if src.resident:
                check_matrix(P)
            else:
                check_matrix(P, r0, None if src.symmetric else src.column_strip(r0, r1))
            core[r0:r1] = kth_smallest(P, ms + 1)
        u, v, w = mutual_reachability_mst(src, core)
        (self.labels_, self.probabilities_, self.condensed_tree_, self.single_linkage_tree_,
         self.minimum_spanning_tree_) = hdbscan_tree(u.cpu().numpy(), v.cpu().numpy(), w.cpu().numpy(), n, self.min_cluster_size)
        return self

    def fit_predict(self, X, y=None):
        return self.fit(X).labels_


TSNE_MAX_K = 1024  # po_matrix_knn's largest k


def check_tsne_matrix(D, row0=0):
    """Refuse (PhyloligoError) a device matrix holding a NaN, an infinite or a negative entry, as scikit-learn's
    TSNE(metric="precomputed") does; the message names the first one in row-major order (po_tsne_check).  With
    row0, D holds the rows [row0, row0 + rows) of the matrix and the message names the absolute entry."""
    lib = _lib.load()
    work = torch.empty(1, dtype=torch.int64, device=D.device)
    rc = lib.po_tsne_check(_ptr(D), int(D.stride(0)), _dt(D), int(D.shape[0]), int(D.shape[1]), int(row0), _ptr(work),
                           _stream())
    _lib.check(rc, "po_tsne_check")


def _fixed_sum(x):
    """float64 sum of a device vector in a fixed order (po_tsne_sum), as a 1-element device tensor."""
    out = torch.empty(1, dtype=torch.float64, device=x.device)
    _lib.check(_lib.load().po_tsne_sum(_ptr(x), int(x.numel()), _ptr(out), _stream()), "po_tsne_sum")
    return out


def tsne_affinities(D, perplexity, as_sparse=False):
    """The joint probabilities P of scikit-learn's TSNE(metric="precomputed", method="barnes_hut") from the device
    matrix D: the k = min(n - 1, int(3 perplexity + 1)) nearest neighbours of every row (po_matrix_knn), their
    squared distances, the per-row perplexity search (po_tsne_conditional), then P = (C + C^T) / sum(C + C^T) with
    the pairs whose sum is 0 dropped, as scipy's sparse addition drops them.  Returns the symmetric CSR as device
    tensors (indptr int64 [n + 1], indices int32, data float64), columns ascending in every row, or with
    `as_sparse` the scipy CSR matrix.  The transpose and the merge of the two halves are torch sort and gather
    plumbing; each merged value is one addition of two terms, and the total is a fixed-order sum, so the result
    is deterministic."""
    src = D if isinstance(D, panels.SOURCES) else panels.ResidentSource(
        D if isinstance(D, torch.Tensor) and D.is_cuda else as_device_matrix(D))
    return _affinities(src, perplexity, as_sparse=as_sparse)


def _affinities(src, perplexity, as_sparse=False, check=False):
    """tsne_affinities over the panels of a source, with `check` the input check of every panel first
    (check_tsne_matrix; the first panel with an offending entry stops the pass)."""
    lib = _lib.load()
    n = src.n
    dev = src.device
    k = min(n - 1, int(3.0 * perplexity + 1))
    for r0, r1, P in src.panels():
        if check:
            check_tsne_matrix(P, r0)
        if r0 == 0:  # after the first panel's check, as the whole-matrix check came first
            if k > TSNE_MAX_K:
                raise ValueError("perplexity {} needs {} neighbours per point; at most {} are supported (perplexity <= 341)"
                                 .format(perplexity, k, TSNE_MAX_K))
            idx = torch.empty((n, k), dtype=torch.int32, device=dev)
            dist = torch.empty((n, k), dtype=torch.float32, device=dev)
            cond = torch.empty((n, k), dtype=torch.float64, device=dev)
        _knn_rows(P, r0, k, idx[r0:r1], dist[r0:r1])
        # po_tsne_conditional takes n as the row count: row i of P is matrix row r0 + i
        rc = lib.po_tsne_conditional(_ptr(P), int(P.stride(0)), _dt(P), r1 - r0, _ptr(idx[r0:r1]), k, float(perplexity),
                                     _ptr(cond[r0:r1]), _stream())
        _lib.check(rc, "po_tsne_conditional")
    rows = torch.arange(n, dtype=torch.int64, device=dev).repeat_interleave(k)
    cols = idx.reshape(-1).to(torch.int64)
    keys, order = torch.sort(torch.cat([rows * n + cols, cols * n + rows]), stable=True)
    vals = torch.cat([cond.reshape(-1), cond.reshape(-1)])[order]
    m = int(keys.numel())
    first = torch.ones(m, dtype=torch.bool, device=dev)
    first[1:] = keys[1:] != keys[:-1]
    starts = torch.nonzero(first).flatten()
    nxt = torch.clamp(starts + 1, max=m - 1)
    paired = (starts + 1 < m) & (keys[nxt] == keys[starts])
    merged = vals[starts] + torch.where(paired, vals[nxt], torch.zeros_like(vals[nxt]))  # C_ij + C_ji (at most two terms)
    keep = merged != 0
    ukeys, data = keys[starts][keep], merged[keep]
    indices = (ukeys % n).to(torch.int32)
    indptr = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    indptr[1:] = torch.cumsum(torch.bincount(ukeys // n, minlength=n), 0)
    total = max(float(_fixed_sum(data).item()), float(np.finfo(np.float64).eps))
    data = data / total
    if not as_sparse:
        return indptr, indices, data
    from scipy.sparse import csr_matrix
    return csr_matrix((data.cpu().numpy(), indices.cpu().numpy(), indptr.cpu().numpy()), shape=(n, n))


def _device_csr(P, device):
    if isinstance(P, tuple):
        return tuple(t.to(device) for t in P)
    P = P.tocsr()
    return (torch.from_numpy(np.asarray(P.indptr, dtype=np.int64)).to(device),
            torch.from_numpy(np.asarray(P.indices, dtype=np.int32)).to(device),
            torch.from_numpy(np.asarray(P.data, dtype=np.float64)).to(device))


class _Descent:
    """Device state of one t-SNE optimisation: two position buffers, update, gains and the workspace."""

    def __init__(self, P, Y0):
        self.lib = _lib.load()
        dev = P[0].device
        self.P = P
        self.n = int(Y0.shape[0])
        self.Y = torch.as_tensor(np.ascontiguousarray(Y0, dtype=np.float32)).to(dev)
        self.Y_next = torch.empty_like(self.Y)
        self.update = torch.zeros((self.n, 2), dtype=torch.float64, device=dev)
        self.gains = torch.ones((self.n, 2), dtype=torch.float32, device=dev)
        self.work = torch.empty(int(self.lib.po_tsne_workspace(self.n)), dtype=torch.uint8, device=dev)
        self.out = (C.c_double * 2)()

    def gradient(self, mul, div, Y_next=None, grad=None, momentum=0.0, lr=0.0, update64=True, compute_error=False):
        lib = self.lib
        _lib.check(lib.po_tsne_repulsion(_ptr(self.Y), self.n, _ptr(self.work), _stream()), "po_tsne_repulsion")
        indptr, indices, data = self.P
        rc = lib.po_tsne_attraction_step(_ptr(indptr), _ptr(indices), _ptr(data), self.n, float(mul), float(div), _ptr(self.Y),
                                         _ptr(self.work), _ptr(Y_next), _ptr(self.update), _ptr(self.gains), _ptr(grad),
                                         float(momentum), float(lr), int(update64), self.out if compute_error else None, _stream())
        _lib.check(rc, "po_tsne_attraction_step")
        return self.out[0], self.out[1]

    def descend(self, it, max_iter, momentum, lr, update64, mul, div, n_iter_without_progress, min_grad_norm, n_iter_check=50):
        """scikit-learn's _gradient_descent: returns (error, last iteration index)."""
        self.update.zero_()
        self.gains.fill_(1.0)
        error = best_error = np.finfo(float).max
        best_iter = i = it
        for i in range(it, max_iter):
            check = (i + 1) % n_iter_check == 0
            compute_error = check or i == max_iter - 1
            kl, gn2 = self.gradient(mul, div, Y_next=self.Y_next, momentum=momentum, lr=lr, update64=update64,
                                    compute_error=compute_error)
            self.Y, self.Y_next = self.Y_next, self.Y
            if compute_error:
                error = kl
            if check:
                if error < best_error:
                    best_error, best_iter = error, i
                elif i - best_iter > n_iter_without_progress:
                    break
                if np.sqrt(gn2) <= min_grad_norm:
                    break
        return error, i


def tsne_gradient(P, Y, exaggeration=1.0):
    """(grad float32 [n, 2], KL) of the t-SNE objective at the positions Y for the joint probabilities P (the
    device CSR of tsne_affinities or a scipy CSR): what scikit-learn's _kl_divergence_bh(angle=0.0) returns with
    P * exaggeration, the repulsion summed exactly over all pairs on the device."""
    dev = engine.require_cuda()
    P = _device_csr(P, dev)
    Y = Y.cpu().numpy() if isinstance(Y, torch.Tensor) else np.asarray(Y)
    st = _Descent(P, Y)
    grad = torch.empty((st.n, 2), dtype=torch.float32, device=dev)
    kl, _ = st.gradient(exaggeration, 1.0, grad=grad, compute_error=True)
    return grad.cpu().numpy(), kl


def _random_state(seed):
    """sklearn.utils.check_random_state"""
    if seed is None or seed is np.random:
        return np.random.mtrand._rand
    if isinstance(seed, (int, np.integer)):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError("%r cannot be used to seed a numpy.random.RandomState instance" % (seed,))


class TSNE:
    """t-SNE on the device: what sklearn.manifold.TSNE(metric="precomputed", method="barnes_hut", angle=0.0)
    computes (scikit-learn 1.9), which with angle 0 is the exact gradient of the sparse-P objective.  Same
    constructor arguments and defaults; ``method``, ``angle``, ``verbose``, ``metric_params`` and ``n_jobs`` are
    accepted at "barnes_hut", 0.0, 0, None and None only.  ``metric`` is "precomputed" (X is the N x N matrix:
    ndarray, memmap or a device tensor, used in place and not modified) or one of the package's metrics (X is the
    N x D profile matrix and the distances never leave the device).  ``init`` is "random" (scikit-learn's draw on
    the host, bit for bit) or an (N, 2) array, used as float32.  Fitted attributes: ``embedding_`` (float32),
    ``kl_divergence_``, ``n_iter_``, ``learning_rate_``."""

    _EXPLORATION_MAX_ITER = 250
    _N_ITER_CHECK = 50
    # scikit-learn's arguments this implementation takes at one value only
    FIXED = {"method": "barnes_hut", "angle": 0.0, "verbose": 0, "metric_params": None, "n_jobs": None}

    def __init__(self, n_components=2, *, perplexity=30.0, early_exaggeration=12.0, learning_rate="auto", max_iter=1000,
                 n_iter_without_progress=300, min_grad_norm=1e-7, metric="precomputed", metric_params=None, init="random",
                 verbose=0, random_state=None, method="barnes_hut", angle=0.0, n_jobs=None):
        given = {"method": method, "angle": angle, "verbose": verbose, "metric_params": metric_params, "n_jobs": n_jobs}
        for key, value in given.items():
            if value is not self.FIXED[key] and value != self.FIXED[key]:
                raise ValueError("{}={!r} is not supported; only {!r} (the exact gradient)".format(key, value, self.FIXED[key]))
        if n_components != 2:
            raise ValueError("n_components={!r} is not supported; only 2".format(n_components))
        if not perplexity > 0:
            raise ValueError("perplexity must be positive, got {!r}".format(perplexity))
        if not early_exaggeration >= 1:
            raise ValueError("early_exaggeration must be at least 1, got {!r}".format(early_exaggeration))
        if not (isinstance(learning_rate, str) and learning_rate == "auto") and not (
                isinstance(learning_rate, (int, float, np.integer, np.floating)) and learning_rate > 0):
            raise ValueError("learning_rate must be 'auto' or positive, got {!r}".format(learning_rate))
        if not isinstance(max_iter, (int, np.integer)) or max_iter < self._EXPLORATION_MAX_ITER:
            raise ValueError("max_iter must be an integer of at least 250, got {!r}".format(max_iter))
        if isinstance(init, str) and init == "pca":
            raise ValueError('The parameter init="pca" cannot be used with metric="precomputed".' if metric == "precomputed"
                             else 'init="pca" is not supported; use "random" or an array')
        if not (isinstance(init, str) and init == "random") and not isinstance(init, np.ndarray):
            raise ValueError("init must be 'random' or an (n_samples, 2) array, got {!r}".format(init))
        if metric != "precomputed" and metric not in _lib.METRICS:
            raise ValueError("metric needs to be 'precomputed' or one of {}. Instead, '{}' was given.".format(sorted(_lib.METRICS), metric))
        self.n_components = n_components
        self.perplexity = perplexity
        self.early_exaggeration = early_exaggeration
        self.learning_rate = learning_rate
        self.max_iter = max_iter
        self.n_iter_without_progress = n_iter_without_progress
        self.min_grad_norm = min_grad_norm
        self.metric = metric
        self.metric_params = metric_params
        self.init = init
        self.verbose = verbose
        self.random_state = random_state
        self.method = method
        self.angle = angle
        self.n_jobs = n_jobs

    def fit_transform(self, X, y=None):
        src = _source(X, self.metric)
        n = src.n
        if n < 2:
            raise ValueError("TSNE needs at least 2 samples, got {}".format(n))
        if self.perplexity >= n:
            raise ValueError("perplexity ({}) must be less than n_samples ({})".format(self.perplexity, n))
        if self.learning_rate == "auto":
            self.learning_rate_ = np.maximum(n / self.early_exaggeration / 4, 50)
        else:
            self.learning_rate_ = self.learning_rate
        P = _affinities(src, self.perplexity, check=True)  # one pass: check, neighbours, conditional P
        if isinstance(self.init, np.ndarray):
            if self.init.shape != (n, 2):
                raise ValueError("init has shape {}; ({}, 2) is expected".format(self.init.shape, n))
            Y0 = self.init
        else:
            Y0 = 1e-4 * _random_state(self.random_state).standard_normal(size=(n, self.n_components)).astype(np.float32)
        st = _Descent(P, Y0)
        # scikit-learn's update is float64 when the learning rate is a float64 scalar ("auto": np.maximum), float32
        # for a Python float
        update64 = (self.learning_rate_ * np.ones(1, np.float32)).dtype == np.float64
        ee, lr = float(self.early_exaggeration), float(self.learning_rate_)
        kl, it = st.descend(0, self._EXPLORATION_MAX_ITER, 0.5, lr, update64, ee, 1.0, self._EXPLORATION_MAX_ITER,
                            self.min_grad_norm, self._N_ITER_CHECK)
        if it < self._EXPLORATION_MAX_ITER or self.max_iter - self._EXPLORATION_MAX_ITER > 0:
            kl, it = st.descend(it + 1, self.max_iter, 0.8, lr, update64, ee, ee, self.n_iter_without_progress, self.min_grad_norm,
                                self._N_ITER_CHECK)
        self.n_iter_ = it
        self.kl_divergence_ = kl
        self.embedding_ = st.Y.cpu().numpy()
        return self.embedding_

    def fit(self, X, y=None):
        self.fit_transform(X)
        return self


LINKAGE_METHODS = {"single": 0, "complete": 1, "average": 2, "weighted": 3, "ward": 4}


def _check_linkage_method(method):
    if method in ("centroid", "median"):
        raise ValueError("method={!r} is not supported: scipy builds it with a different algorithm (the Lance-Williams "
                         "update is not reducible there); use one of {}".format(method, list(LINKAGE_METHODS)))
    if method not in LINKAGE_METHODS:
        raise ValueError("method must be one of {}, got {!r}".format(list(LINKAGE_METHODS), method))


def linkage_bytes(n, method):
    """Device bytes linkage(D, method) allocates for n rows besides D: the float64 n x n working copy (not for
    "single", which reads D in place), the workspace and the raw merges."""
    _check_linkage_method(method)
    return int(_lib.load().po_linkage_workspace(n)) + 24 * (n - 1) + (0 if method == "single" else 8 * n * n)


def check_linkage_fits(n, method, free_bytes):
    """Refuse (PhyloligoError) a linkage of n rows whose device memory (linkage_bytes) exceeds free_bytes."""
    need = linkage_bytes(n, method)
    if need > free_bytes:
        raise PhyloligoError("linkage(method={!r}) of {} rows needs {} bytes of device memory ({}), {} are free".format(
            method, n, need, "the float64 working copy of the matrix and the workspace" if method != "single" else "the workspace",
            free_bytes))


def linkage_raw(D, method="average"):
    """The n - 1 merges of scipy's nn_chain (Prim for "single") on the device matrix D, in merge order, before the
    sort and relabelling: device tensors (x int64, y int64, height float64) and the number of grid barriers the
    launch took (po_linkage_run).  D is checked (check_matrix) and not modified."""
    _check_linkage_method(method)
    lib = _lib.load()
    n = int(D.shape[0])
    if n < 2:
        raise ValueError("linkage needs at least 2 observations, got {}".format(n))
    check_matrix(D)
    dev = D.device
    free, _ = torch.cuda.mem_get_info(dev)
    free += torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
    check_linkage_fits(n, method, free)
    W = None if method == "single" else torch.empty((n, n), dtype=torch.float64, device=dev)
    work = torch.empty(int(lib.po_linkage_workspace(n)), dtype=torch.uint8, device=dev)
    zx = torch.empty(n - 1, dtype=torch.int64, device=dev)
    zy = torch.empty_like(zx)
    zh = torch.empty(n - 1, dtype=torch.float64, device=dev)
    phases = C.c_int64()
    rc = lib.po_linkage_run(_ptr(D), int(D.stride(0)), _dt(D), n, LINKAGE_METHODS[method], _ptr(W), _ptr(work), _ptr(zx), _ptr(zy),
                            _ptr(zh), C.byref(phases), _stream())
    _lib.check(rc, "po_linkage_run")
    return zx, zy, zh, phases.value


def linkage_tree(x, y, h):
    """Host stage (po_linkage_tree): the stable sort of the raw merges by height and scipy's label, giving the
    (n - 1, 4) linkage matrix."""
    x = np.ascontiguousarray(x, dtype=np.int64)
    y = np.ascontiguousarray(y, dtype=np.int64)
    h = np.ascontiguousarray(h, dtype=np.float64)
    n = len(x) + 1
    Z = np.empty((n - 1, 4), dtype=np.float64)
    rc = _lib.load().po_linkage_tree(n, *[C.c_void_p(a.ctypes.data) for a in (x, y, h, Z)])
    _lib.check(rc, "po_linkage_tree")
    return Z


def linkage(D, method="average"):
    """Hierarchical clustering on the device: the (n - 1, 4) float64 array that
    scipy.cluster.hierarchy.linkage(squareform(D, checks=False), method) returns, bit for bit, for method "single",
    "complete", "average", "weighted" or "ward".  D is an ndarray, a memmap or a device tensor (used in place and
    not modified); it must be square, bitwise symmetric and finite.  All but "single" use a float64 working copy of
    D on the device (8 n^2 bytes); a matrix whose copy does not fit is refused before anything is allocated."""
    _check_linkage_method(method)
    D = as_device_matrix(D)
    x, y, h, _ = linkage_raw(D, method)
    return linkage_tree(x.cpu().numpy(), y.cpu().numpy(), h.cpu().numpy())


class HClust:
    """The tree phyloselect.R builds with hclust, cut into flat clusters.  ``linkage_`` is Z (see linkage) and
    ``labels_`` = scipy.cluster.hierarchy.fcluster(Z, n_clusters, "maxclust") - 1, numbered from 0 as KMedoids'
    labels are (fewer than n_clusters clusters when heights tie, as scipy gives).  ``metric`` is "precomputed" (X
    is the N x N matrix: ndarray, memmap or a device tensor, used in place) or one of the package's metrics (X is
    the N x D profile matrix and the distances never leave the device)."""

    def __init__(self, n_clusters=8, linkage="average", metric="precomputed"):
        if not isinstance(n_clusters, (int, np.integer)) or isinstance(n_clusters, bool) or n_clusters < 1:
            raise ValueError("n_clusters must be a positive integer, got {!r}".format(n_clusters))
        _check_linkage_method(linkage)
        if metric != "precomputed" and metric not in _lib.METRICS:
            raise ValueError("metric needs to be 'precomputed' or one of {}. Instead, '{}' was given.".format(sorted(_lib.METRICS), metric))
        self.n_clusters = int(n_clusters)
        self.linkage = linkage
        self.metric = metric

    def fit(self, X, y=None):
        from scipy.cluster.hierarchy import fcluster
        if self.metric == "precomputed":
            D = X
        else:
            Xd = X if isinstance(X, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(np.asarray(X)))
            D = engine.distance_matrix_device(Xd.to(engine.require_cuda()), self.metric, torch.float32, symmetric=True)
        self.linkage_ = linkage(D, self.linkage)
        self.labels_ = fcluster(self.linkage_, self.n_clusters, "maxclust").astype(np.int64) - 1
        return self

    def fit_predict(self, X, y=None):
        return self.fit(X).labels_


NJ_METHODS = {"nj": 0, "bionj": 1}


def _check_nj_method(method):
    if method not in NJ_METHODS:
        raise ValueError("method must be one of {}, got {!r}".format(list(NJ_METHODS), method))


def nj_bytes(n, method="nj"):
    """Device bytes nj(D, method) allocates for n rows besides D: the float64 C x C working state (C = n plus a front
    headroom of new-node slots, po_nj_capacity; BIONJ keeps its variance in the same array, below the diagonal), the
    compaction's staging rows, the workspace and the edges."""
    _check_nj_method(method)
    lib = _lib.load()
    c = int(lib.po_nj_capacity(n))
    return 8 * c * c + int(lib.po_nj_stage_bytes(n)) + int(lib.po_nj_workspace(n)) + 24 * (2 * n - 3)


def check_nj_fits(n, method, free_bytes):
    """Refuse (PhyloligoError) a tree of n rows whose device memory (nj_bytes) exceeds free_bytes."""
    need = nj_bytes(n, method)
    if need > free_bytes:
        raise PhyloligoError("nj(method={!r}) of {} rows needs {} bytes of device memory (the float64 working state of "
                             "the matrix, the staging rows and the workspace), {} are free".format(method, n, need, free_bytes))


def nj_raw(D, method="nj"):
    """nj on the device matrix D: device tensors (edge int64 (2n - 3, 2), length float64 (2n - 3,)) and the number
    of compactions of the working state (po_nj_run).  D is checked (check_matrix) and not modified."""
    _check_nj_method(method)
    lib = _lib.load()
    n = int(D.shape[0])
    if n < 3:
        raise ValueError("nj needs at least 3 observations, got {}".format(n))
    check_matrix(D)
    dev = D.device
    free, _ = torch.cuda.mem_get_info(dev)
    free += torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
    check_nj_fits(n, method, free)
    c = int(lib.po_nj_capacity(n))
    W = torch.empty((c, c), dtype=torch.float64, device=dev)
    stage = torch.empty(int(lib.po_nj_stage_bytes(n)), dtype=torch.uint8, device=dev)
    work = torch.empty(int(lib.po_nj_workspace(n)), dtype=torch.uint8, device=dev)
    edge = torch.empty((2 * n - 3, 2), dtype=torch.int64, device=dev)
    length = torch.empty(2 * n - 3, dtype=torch.float64, device=dev)
    compactions = C.c_int64()
    rc = lib.po_nj_run(_ptr(D), int(D.stride(0)), _dt(D), n, NJ_METHODS[method], _ptr(W), _ptr(stage), _ptr(work), _ptr(edge),
                       _ptr(length), C.byref(compactions), _stream())
    _lib.check(rc, "po_nj_run")
    return edge, length, compactions.value


def nj(D, method="nj"):
    """Neighbour joining on the device: the unrooted tree phyloselect.R builds with ape's ``nj`` (method "nj") or
    ``bionj`` ("bionj"), in the order of float64 operations DESIGN.md section 4.11 fixes, bit for bit.  Agreement with ape itself is
    not pinned: ape's C source has not been available to compare against, and its bionj is Gascuel's own program,
    whose pair order and tie tolerance are not restated.  D is an ndarray, a memmap or a device tensor, float32 or
    float64 (float32 is widened exactly), used in place and not modified; it must be square, bitwise symmetric and
    finite.  Returns (edge int64 (2n - 3, 2) of (parent, child), length float64 (2n - 3,)) in ape's numbering from
    0: leaves 0 .. n-1, the root n, the node of join t (t = 0, 1, ...) 2n - 3 - t.  Rows are in join order, the
    first-listed member first, then the three root edges in list order.  A working state (8 C^2 bytes, C slightly
    above n) that does not fit in device memory is refused before anything is allocated."""
    _check_nj_method(method)
    D = as_device_matrix(D)
    edge, length, _ = nj_raw(D, method)
    return edge.cpu().numpy(), length.cpu().numpy()


def write_nj_newick(edge, length, names, path):
    """Write the tree of nj (edge, length) as an unrooted Newick tree with leaves names[0 .. n), shaped as ape's
    write.tree writes it: a trifurcating root whose children are the root edges in order, every joined node's two
    children in join order.  Lengths are repr(float), names go through newick_name.  The walk is iterative:
    caterpillar trees are n deep."""
    edge = np.asarray(edge, dtype=np.int64)
    length = np.asarray(length, dtype=np.float64)
    n = (len(edge) + 3) // 2
    if edge.ndim != 2 or edge.shape != (2 * n - 3, 2) or length.shape != (2 * n - 3,) or n < 3 or len(names) != n:
        raise ValueError("a ({0}, 2) edge matrix, {0} lengths and {1} names are expected, got {2}, {3} and {4} names".format(
            2 * n - 3, n, edge.shape, length.shape, len(names)))
    children = {}
    for (parent, child), ln in zip(edge.tolist(), length.tolist()):
        children.setdefault(parent, []).append((child, ln))
    out = []
    stack = [(n, "")]
    while stack:
        item = stack.pop()
        if isinstance(item, str):
            out.append(item)
            continue
        node, tail = item
        if node < n:
            out.append(newick_name(names[node]) + tail)
            continue
        out.append("(")
        stack.append(")" + tail)
        kids = children[node]
        for i in range(len(kids) - 1, -1, -1):
            child, ln = kids[i]
            stack.append((child, ":" + repr(float(ln))))
            if i:
                stack.append(",")
    with open(path, "w") as fh:
        fh.write("".join(out) + ";\n")


def newick_name(name):
    """A Newick leaf label: single-quoted, with every ' doubled, when it is empty or holds a blank or one of
    ( ) [ ] ' : ; ,"""
    s = str(name)
    if s == "" or any(c in "()[]':;," or c.isspace() for c in s):
        return "'" + s.replace("'", "''") + "'"
    return s


def write_newick(Z, names, path):
    """Write the linkage matrix Z as a rooted Newick tree with leaves names[0 .. n).  Node depth is height / 2
    (the ultrametric convention of ape's as.phylo(hclust)), so a leaf-to-leaf path is as long as the height of the
    two leaves' merge.  Children are written in Z's order (column 0, then column 1).  The walk is iterative:
    single-linkage trees can be n deep."""
    Z = np.asarray(Z, dtype=np.float64)
    n = Z.shape[0] + 1
    if Z.ndim != 2 or Z.shape[1] != 4 or len(names) != n:
        raise ValueError("a ({}, 4) linkage matrix and {} names are expected, got {} and {} names".format(n - 1, n, Z.shape, len(names)))
    depth = Z[:, 2] / 2.0

    def length(child, parent_depth):
        return repr(float(parent_depth - (depth[child - n] if child >= n else 0.0)))

    out = []
    stack = [(2 * n - 2, "")]
    while stack:
        item = stack.pop()
        if isinstance(item, str):
            out.append(item)
            continue
        node, tail = item
        if node < n:
            out.append(newick_name(names[node]) + tail)
            continue
        k = node - n
        a, b = int(Z[k, 0]), int(Z[k, 1])
        out.append("(")
        stack += [")" + tail, (b, ":" + length(b, depth[k])), ",", (a, ":" + length(a, depth[k]))]
    with open(path, "w") as fh:
        fh.write("".join(out) + ";\n")


# ---------------------------------------------------------------------------
# the script's functions
# ---------------------------------------------------------------------------
def read_distmat(path):
    """reference :357-371"""
    return np.loadtxt(path)


def read_matrix(path, large=False):
    """The three on-disk conventions of phyloligo.py (reference main :601-622)."""
    if large == "memmap":
        matrix = np.memmap(path, dtype=np.float32, mode="r")
        n = int(round(np.sqrt(matrix.shape[0])))
        if n * n != matrix.shape[0]:
            print("Error, weird shape for matrix {}".format(path), file=sys.stderr)
            sys.exit(1)
        return matrix.reshape((n, n))
    if large == "h5py":
        return io_formats.read_hdf5(path, "distances")
    return read_distmat(path)


def read_source(path, large=False):
    """The matrix of `path` for the clustering methods: resident on the device when it fits with their working
    state (panels.fits), else, for a --large memmap / h5py file, a panels.FileSource that reads it panel by panel
    (never the whole file into host memory).  A text matrix that does not fit is refused with its byte count."""
    if large:
        if large == "memmap":
            size = os.path.getsize(path) // 4
            n = int(round(np.sqrt(size)))
            if n * n != size:
                print("Error, weird shape for matrix {}".format(path), file=sys.stderr)
                sys.exit(1)
            offset, dtype = 0, np.float32
        else:
            shape, dtype, offset = io_formats.dataset_location(path, "distances")
            if len(shape) != 2 or shape[0] != shape[1]:
                raise PhyloligoError("a square distance matrix is expected, got shape %s" % (tuple(shape),))
            n = int(shape[0])
        if panels.fits(n, np.dtype(dtype).itemsize):
            return panels.ResidentSource(as_device_matrix(read_matrix(path, large)))
        return panels.FileSource(path, n, offset=offset, dtype=dtype)
    matrix = read_matrix(path, large)
    n = int(matrix.shape[0]) if matrix.ndim == 2 else 0
    budget = panels.device_budget()
    if not panels.fits(n, 8, budget):
        raise PhyloligoError("a text matrix of {} rows needs {} bytes of device memory (float64, with the working state), "
                             "{} are free; write it with phyloligo.py --large memmap or h5py to cluster it in row panels"
                             .format(n, 8 * n * n + panels.state_bytes(n), budget))
    return panels.ResidentSource(as_device_matrix(matrix))


def check_resident_methods(params, n, element_size):
    """Refuse (PhyloligoError), before any pass, what needs the matrix resident: -m hclust and --tree-out keep an
    O(n^2) float64 working state besides it."""
    wants = (["-m hclust"] if params.method == "hclust" else []) + (["--tree-out"] if params.tree_out else [])
    if not wants:
        return
    budget = panels.device_budget()
    work = nj_bytes(n, params.tree_method) if params.tree_out and params.tree_method != "hclust" else linkage_bytes(n, params.linkage)
    need = int(n) * int(n) * int(element_size) + work
    raise PhyloligoError("{} of {} rows needs {} bytes of device memory (the matrix and the tree's float64 working state), "
                         "{} are free".format(" and ".join(wants), n, need, budget))


def find_clusters(data, method, kwargs, return_model=False):
    """reference :403-428; with `return_model` the fitted estimator (its ``labels_`` are what is returned
    otherwise; HClust's also holds the tree, ``linkage_``)"""
    if method == "kmedoids":
        model = KMedoids(**kwargs)
    elif method == "hdbscan":
        model = HDBSCAN(**kwargs)
    elif method == "hclust":
        model = HClust(**kwargs)
    else:
        print("Error, unknown method {}".format(method), file=sys.stderr)
        sys.exit(1)
    model.fit(data)
    return model if return_model else model.labels_


def clusterize(data, method, min_cluster_size=None, min_samples=None, nbk=None, linkage_method=None, return_model=False):
    """reference :573-590"""
    kwargs = dict()
    if method == "hclust":
        if nbk is not None:
            kwargs["n_clusters"] = nbk
        if linkage_method is not None:
            kwargs["linkage"] = linkage_method
        kwargs["metric"] = "precomputed"
    if method == "hdbscan":
        if min_cluster_size is not None:
            kwargs["min_cluster_size"] = min_cluster_size
        if min_samples is not None:
            kwargs["min_samples"] = min_samples
        kwargs["metric"] = "precomputed"
    if method == "kmedoids":
        if nbk is not None:
            kwargs["n_clusters"] = nbk
        kwargs["distance_metric"] = "precomputed"
    return find_clusters(data, method, kwargs, return_model=return_model)


def write_cluster_indexes(labels_pred, pathout):
    """``data_cluster_indexes.dat``: one "class index" line per contig, grouped by class (reference :742-751)."""
    labels_pred = np.asarray(labels_pred)
    with open(pathout, "w") as outf:
        for cl in np.unique(labels_pred):
            for idx in np.where(labels_pred == cl)[0]:
                outf.write("{} {}\n".format(cl, idx))


def write_fastafile(labels_pred, fastafile, outputdir):
    """One FASTA file per class, ``data_fasta_cl{c}.fa`` / ``data_fasta_unclust.fa`` (reference :547-571).
    Records are written as Biopython's SeqIO.write does: the title line unchanged, the sequence wrapped at
    60 columns."""
    labels_pred = np.asarray(labels_pred)
    text = np.fromfile(fastafile, dtype=np.uint8)
    begin, end = engine.fasta_index(text)
    if len(begin) != len(labels_pred):
        raise PhyloligoError("{} holds {} records, the matrix {} rows".format(fastafile, len(begin), len(labels_pred)))
    raw = text.tobytes()
    starts = engine.fasta_header_starts(raw, begin, end)
    for cl in np.unique(labels_pred):
        name = "data_fasta_unclust.fa" if cl == -1 else "data_fasta_cl{}.fa".format(cl)
        with open(os.path.join(outputdir, name), "wb") as outf:
            for idx in np.where(labels_pred == cl)[0]:
                b, e = int(begin[idx]), int(end[idx])
                title = raw[int(starts[idx]):b].rstrip(b"\r\n")
                seq = b"".join(raw[b:e].split())
                outf.write(title + b"\n")
                for p in range(0, len(seq), 60):
                    outf.write(seq[p:p + 60] + b"\n")


def fasta_record_ids(fastafile):
    """The id of every record of a FASTA file: its title up to the first blank."""
    text = np.fromfile(fastafile, dtype=np.uint8)
    begin, end = engine.fasta_index(text)
    raw = text.tobytes()
    ids = []
    for s, b in zip(engine.fasta_header_starts(raw, begin, end), begin):
        title = raw[int(s):int(b)].strip()
        title = title[1:] if title.startswith(b">") else title
        ids.append((title.split(None, 1) or [b""])[0].decode("utf-8", "replace"))
    return ids


def get_cmd(argv=None):
    parser = argparse.ArgumentParser(description="Cluster contigs from their oligonucleotide-profile distances on B200 GPUs")
    parser.add_argument("-i", action="store", dest="distmat", help="The input matrix file")
    parser.add_argument("-m", action="store", dest="method", required=True, choices=["hdbscan", "kmedoids", "hclust"],
                        help="Method to use to compute cluster on the distance matrix: HDBSCAN (--minclustersize, "
                             "--minsamples; noise goes to data_fasta_unclust.fa), K-medoids (-k) or the hierarchical "
                             "tree cut into -k clusters (--linkage)")
    parser.add_argument("--minclustersize", action="store", dest="min_cluster_size", type=int,
                        help="Set the minimal cluster size of an HDBSCAN cluster")
    parser.add_argument("--minsamples", action="store", dest="min_samples", type=int,
                        help="Set the minimal sample size of an HDBSCAN cluster")
    parser.add_argument("-k", action="store", dest="nbk", type=int, help="Number of cluster")
    parser.add_argument("--linkage", action="store", dest="linkage", default="average", choices=list(LINKAGE_METHODS),
                        help="linkage of -m hclust and --tree-out (scipy.cluster.hierarchy.linkage's method)")
    parser.add_argument("--tree-out", action="store", dest="tree_out",
                        help="write the tree of the matrix (--tree-method) to this file in Newick format; leaves "
                             "are the FASTA record ids with -f or --assembly, row indices otherwise")
    parser.add_argument("--tree-method", action="store", dest="tree_method", default="hclust", choices=["hclust"] + list(NJ_METHODS),
                        help="the tree --tree-out writes: the hierarchical tree (hclust, --linkage, rooted) or the "
                             "neighbour-joining tree (nj, bionj: ape's nj / bionj as phyloselect.R offers them, unrooted)")
    parser.add_argument("-f", action="store", dest="fastafile",
                        help="Path of the original fasta file used for the computation of the distance matrix")
    parser.add_argument("--large", action="store", choices=["memmap", "h5py"], dest="large", default=False,
                        help="Format of a matrix written with phyloligo.py --large")
    parser.add_argument("-o", action="store", dest="outputdir", required=True)
    parser.add_argument("-t", action="store_true", dest="performtsne", default=False,
                        help="(not built: plotting is out of scope; --tsne-out writes the embedding)")
    parser.add_argument("--interactive", action="store_true", dest="interactive", default=False,
                        help="(not built: plotting is out of scope)")
    parser.add_argument("--noX", action="store_true", dest="noX", help="accepted for compatibility")
    parser.add_argument("-p", action="store", dest="perplexity", default=100, type=int, help="t-SNE perplexity (--tsne-out)")
    parser.add_argument("--tsne-out", action="store", dest="tsne_out",
                        help="write the 2-D t-SNE embedding of the matrix (perplexity -p, random_state 0) to this file: one "
                             "tab-separated %%.18e row per contig")
    parser.add_argument("-q", "--infreq", action="store", dest="in_freq_file", help="accepted for compatibility")
    # without a matrix file: profile the assembly and keep the matrix on the device
    parser.add_argument("--assembly", action="store", dest="assembly",
                        help="instead of -i: compute the matrix from this multi-FASTA on the device (no matrix file at all)")
    parser.add_argument("--pattern", action="store", dest="pattern", default="1111", help="spaced-word pattern for --assembly")
    parser.add_argument("--strand", action="store", dest="strand", default="both", choices=["both", "plus", "minus"])
    parser.add_argument("-d", "--distance", action="store", dest="dist", default="JSD", choices=["Eucl", "JSD", "KT", "BC", "SC"])
    params = parser.parse_args(argv)
    if params.performtsne or params.interactive:
        print("Error, t-SNE projection and the interactive mode draw pictures: not part of the GPU front half "
              "(--tsne-out FILE writes the 2-D t-SNE embedding computed on the device)", file=sys.stderr)
        sys.exit(1)
    if not params.distmat and not params.assembly:
        print("Error, give a matrix (-i) or an assembly (--assembly)", file=sys.stderr)
        sys.exit(1)
    return params


def main(argv=None):
    params = get_cmd(argv)
    if not os.path.isdir(params.outputdir):
        os.makedirs(params.outputdir)
    if params.assembly:
        print("Compute matrix")
        from . import phyloligo
        res, n, _ = phyloligo._profile_file(params.assembly, params.pattern, params.strand, ("freq32",))
        if res is None:
            print("Error, no FASTA record in {}".format(params.assembly), file=sys.stderr)
            sys.exit(1)
        source = panels.profile_source(res["freq32"], phyloligo._large_metric(params.dist))
        if params.fastafile is None:
            params.fastafile = params.assembly
    else:
        print("Read matrix")
        source = read_source(params.distmat, params.large)
    if source.resident:
        matrix = source.D
    else:
        check_resident_methods(params, source.n, torch.empty(0, dtype=source.dtype).element_size())
        matrix = source
        print("The matrix does not fit on the device: {} rows in panels of {}".format(source.n, source.panel_rows))
    print("Clusterize")
    model = clusterize(matrix, params.method, min_cluster_size=params.min_cluster_size, min_samples=params.min_samples,
                       nbk=params.nbk, linkage_method=params.linkage, return_model=True)
    labels_pred = model.labels_
    Z = getattr(model, "linkage_", None)  # -m hclust: the tree --tree-out writes
    pathout = os.path.join(params.outputdir, "data_cluster_indexes.dat")
    print("Store cluster indexes in {}".format(pathout))
    write_cluster_indexes(labels_pred, pathout)
    if params.fastafile:
        print("Write fasta per classes in {}/data_fasta_*.fa".format(params.outputdir))
        write_fastafile(labels_pred, params.fastafile, params.outputdir)
    if params.tsne_out:
        print("Store t-SNE embedding in {}".format(params.tsne_out))
        np.savetxt(params.tsne_out, TSNE(perplexity=params.perplexity, random_state=0).fit(matrix).embedding_, delimiter="\t")
    if params.tree_out and params.tree_method != "hclust":
        print("Store the {} tree in {}".format(params.tree_method, params.tree_out))
        edge, length = nj(matrix, params.tree_method)
        n = (len(edge) + 3) // 2
        names = fasta_record_ids(params.fastafile) if params.fastafile else [str(i) for i in range(n)]
        if len(names) != n:
            raise PhyloligoError("{} holds {} records, the matrix {} rows".format(params.fastafile, len(names), n))
        write_nj_newick(edge, length, names, params.tree_out)
    elif params.tree_out:
        print("Store the {} linkage tree in {}".format(params.linkage, params.tree_out))
        if Z is None:
            Z = linkage(matrix, params.linkage)
        names = fasta_record_ids(params.fastafile) if params.fastafile else [str(i) for i in range(Z.shape[0] + 1)]
        if len(names) != Z.shape[0] + 1:
            raise PhyloligoError("{} holds {} records, the matrix {} rows".format(params.fastafile, len(names), Z.shape[0] + 1))
        write_newick(Z, names, params.tree_out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
