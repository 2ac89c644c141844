"""GPU parity of the phyloselect front half (phyloligo_b200/phyloselect.py, csrc/po_select.cu) against the
goldens of the reference's own KMedoids class, the numpy oracle and scikit-learn's neighbour graph."""
import math
import os
import warnings

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle import phylo_oracle as po
from oracle import select_oracle as so
from phyloligo_b200 import engine, io_formats, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(GOLDEN, "select_golden.npz")))


def test_kmedoids_matches_the_reference_goldens(golden):
    for name in golden["names"]:
        D = golden[name + "_D"]
        kw = dict(eval(str(golden[name + "_kwargs"])))
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            km = phyloselect.KMedoids(distance_metric="precomputed", **kw).fit(D)
        assert np.array_equal(km.labels_, golden[name + "_labels"]), name
        assert km.n_iter_ == int(golden[name + "_n_iter"]), name
        assert np.array_equal(km.cluster_centers_, D[golden[name + "_medoids"]]), name
        assert np.array_equal(D[km.medoid_indices_], D[golden[name + "_medoids"]]), name
        assert sum("is empty" in str(w.message) for w in caught) == int(golden[name + "_empty_warnings"]), name


@pytest.mark.parametrize("n,k,dtype", [(1000, 4, np.float32), (2500, 7, np.float64), (333, 1, np.float32), (64, 64, np.float64)])
def test_kmedoids_matches_the_oracle_on_larger_matrices(n, k, dtype):
    rng = np.random.default_rng(n + k)
    centres = rng.normal(0, 4, size=(max(2, k), 6))
    P = centres[rng.integers(0, len(centres), n)] + rng.normal(0, 1, size=(n, 6))
    D = np.sqrt(((P[:, None, :] - P[None, :, :]) ** 2).sum(-1)).astype(dtype)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        labels, medoids, n_iter = so.kmedoids_fit(D.astype(np.float64), n_clusters=k)
        km = phyloselect.KMedoids(n_clusters=k).fit(D)
    assert km.n_iter_ == n_iter and np.array_equal(km.medoid_indices_, medoids) and np.array_equal(km.labels_, labels)
    # a device tensor is used in place, and the row sums are float64 sums of the stored entries
    Dd = torch.from_numpy(D).cuda()
    assert np.allclose(phyloselect.row_sums(Dd).cpu().numpy(), D.astype(np.float64).sum(axis=1), rtol=1e-12)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert np.array_equal(phyloselect.KMedoids(n_clusters=k).fit(Dd).labels_, labels)


def test_kmedoids_from_profiles_never_leaves_the_device():
    seqs = synth.make_sequences(400, 5000, seed=44)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs]).astype(np.float32)
    km = phyloselect.KMedoids(n_clusters=2, distance_metric="JSD").fit(X)
    D = po.pairwise_np(X.astype(np.float64), "JSD")
    labels, medoids, _ = so.kmedoids_fit(D, n_clusters=2)
    assert np.array_equal(km.medoid_indices_, medoids) and np.array_equal(km.labels_, labels)
    assert np.array_equal(km.cluster_centers_, X[medoids])
    with pytest.raises(ValueError):
        phyloselect.KMedoids(n_clusters=2, distance_metric="cosine").fit(X)
    with pytest.raises(ValueError):
        phyloselect.KMedoids(n_clusters=0).fit(D)


KNN_SKLEARN_SHAPES = [(50, 1), (700, 15), (3000, 90), (1200, 300), (40, 39)]


# float32 cases keep their ids ("n-k"), float64 ones add "-float64"
@pytest.mark.parametrize("n,k,dtype", [pytest.param(n, k, np.float32, id="%d-%d" % (n, k)) for n, k in KNN_SKLEARN_SHAPES] +
                         [pytest.param(n, k, np.float64, id="%d-%d-float64" % (n, k)) for n, k in KNN_SKLEARN_SHAPES])
def test_knn_graph_matches_sklearn(n, k, dtype):
    rng = np.random.default_rng(n * 7 + k)
    P = rng.random((n, 4))
    D = np.sqrt(((P[:, None, :] - P[None, :, :]) ** 2).sum(-1)).astype(dtype)
    idx, dist = phyloselect.knn_graph(torch.from_numpy(D).cuda(), k)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    ref_idx, ref_dist = so.knn_graph(D.astype(np.float64), k)
    assert np.array_equal(dist, ref_dist.astype(np.float32))
    assert np.array_equal(dist, np.take_along_axis(D, idx.astype(np.int64), axis=1).astype(np.float32))
    assert (idx != np.arange(n)[:, None]).all() and all(len(set(r)) == k for r in idx.tolist())
    same = idx == ref_idx  # equal distances may be ordered differently by sklearn; ours: ties by column
    assert same.mean() > 0.99
    ties = ~same
    assert np.array_equal(dist[ties], ref_dist.astype(np.float32)[ties])
    # sparse form for TSNE(metric="precomputed"); block rows with the row's own column excluded
    G = phyloselect.knn_graph(D, k, as_sparse=True)
    assert G.shape == (n, n) and G.nnz == n * k
    r0 = n // 3
    bidx, bdist = phyloselect.knn_graph(torch.from_numpy(D[r0:r0 + 17]).cuda(), k, row0=r0)
    assert np.array_equal(bidx.cpu().numpy(), idx[r0:r0 + 17]) and np.array_equal(bdist.cpu().numpy(), dist[r0:r0 + 17])


def test_knn_ties_go_by_column_and_nan_sorts_last():
    D = np.ones((9, 9), dtype=np.float32)
    np.fill_diagonal(D, 0.0)
    D[0, 5] = np.nan
    D[0, 7] = 0.5
    idx, dist = phyloselect.knn_graph(D, 4)
    idx = idx.cpu().numpy()
    assert idx[0].tolist() == [7, 1, 2, 3] and idx[4].tolist() == [0, 1, 2, 3] and idx[8].tolist() == [0, 1, 2, 3]
    with pytest.raises(Exception):
        phyloselect.knn_graph(D, 9)


WIDE_ROW_KINDS = ["smooth", "quantised", "runs", "nan_rows"]


@pytest.mark.parametrize("kind,dtype", [pytest.param(kind, np.float32, id=kind) for kind in WIDE_ROW_KINDS] +
                         [pytest.param(kind, np.float64, id=kind + "-float64") for kind in WIDE_ROW_KINDS])
def test_knn_wide_rows_sampled_threshold_and_fallback(kind, dtype):
    """Rows longer than the 8192-entry sample: the one-pass threshold path, and the rows that must fall back
    to the exact five-pass select (thousands of ties at the threshold, small values hidden between the sampled
    runs, rows that are mostly NaN).  Expected: stable argsort of the row with its own column removed."""
    rng = np.random.default_rng(11)
    rows, n, k, r0 = 24, 30000, 301, 100
    D = rng.random((rows, n), dtype=np.float32)
    if kind == "quantised":
        D = np.floor(D * 4.0).astype(np.float32)  # 7500 ties per level
    elif kind == "runs":
        D += 1.0
        D[:, 200:200 + 2 * k] = rng.random((rows, 2 * k), dtype=np.float32)  # all k smallest in one stretch
        D[5, :] = 2.0
        D[5, 29000:29000 + k + 3] = np.arange(k + 3, dtype=np.float32)[::-1] / 1000.0
    elif kind == "nan_rows":
        D[::2, 400:] = np.nan
        D[3, :] = np.nan
    D = D.astype(dtype)
    idx, dist = phyloselect.knn_graph(torch.from_numpy(D).cuda(), k, row0=r0)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    for i in range(rows):
        row = D[i].astype(np.float64)
        key = np.where(np.isnan(row), np.inf, row)
        order = np.lexsort((np.arange(n), np.isnan(row), key))
        order = order[order != r0 + i][:k]
        assert np.array_equal(idx[i], order), (kind, i)
        assert np.array_equal(dist[i], D[i][order].astype(np.float32), equal_nan=True), (kind, i)


def test_command_line_front_half(tmp_path, capsys):
    seqs = synth.make_sequences(150, 3000, seed=9)
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs])
    D = po.pairwise_np(X, "JSD")
    want, _, _ = so.kmedoids_fit(D, n_clusters=3)
    outs = {}
    np.savetxt(os.path.join(tmp_path, "m.txt"), D, delimiter="\t")
    D.astype(np.float32).tofile(os.path.join(tmp_path, "m.bin"))
    io_formats.write_hdf5(os.path.join(tmp_path, "m.h5"), "distances", D.astype(np.float32))
    for tag, args in (("txt", ["-i", os.path.join(tmp_path, "m.txt")]),
                      ("memmap", ["-i", os.path.join(tmp_path, "m.bin"), "--large", "memmap"]),
                      ("h5py", ["-i", os.path.join(tmp_path, "m.h5"), "--large", "h5py"]),
                      ("device", ["--assembly", fasta, "-d", "JSD", "--pattern", "1111"])):
        out = os.path.join(tmp_path, "out_" + tag)
        assert phyloselect.main(args + ["-m", "kmedoids", "-k", "3", "-o", out, "-f", fasta]) == 0
        rows = [tuple(int(v) for v in line.split()) for line in open(os.path.join(out, "data_cluster_indexes.dat"))]
        labels = np.empty(len(seqs), dtype=np.int64)
        for cl, idx in rows:
            labels[idx] = cl
        outs[tag] = labels
        assert rows == sorted(rows)  # grouped by class, indices ascending (reference :742-751)
        # one FASTA per class, records in file order, sequences intact
        for cl in np.unique(labels):
            recs = open(os.path.join(out, "data_fasta_cl%d.fa" % cl)).read().split(">")[1:]
            members = np.where(labels == cl)[0]
            assert len(recs) == len(members)
            for rec, idx in zip(recs, members):
                lines = rec.split("\n")
                assert lines[0] == "c%d" % idx and "".join(lines[1:]) == seqs[idx].decode()
                assert max(len(l) for l in lines[1:]) <= 60
    assert np.array_equal(outs["txt"], want)
    # float32 files: the same partition unless a cost comparison is within float32 rounding (not here)
    for tag in ("memmap", "h5py", "device"):
        assert np.array_equal(outs[tag], want), tag
    assert "Clusterize" in capsys.readouterr().out
    with pytest.raises(SystemExit):
        phyloselect.main(["-i", "x", "-m", "kmedoids", "-o", str(tmp_path), "-t"])


def test_command_line_against_the_unmodified_reference_scripts(tmp_path):
    """The matrices written by the reference's unmodified bin/phyloligo.py, clustered by its unmodified
    bin/phyloselect.py (tests/golden/make_select_cli_golden.py): this command line on the same matrix files gives
    the same data_cluster_indexes.dat and the same per-cluster FASTA files, byte for byte."""
    import sys
    sys.path.insert(0, GOLDEN)
    import make_cli_golden as mk
    golden = dict(np.load(os.path.join(GOLDEN, "select_cli_golden.npz")))
    fasta, n = mk.assembly()
    path = os.path.join(tmp_path, "asm.fasta")
    open(path, "wb").write(fasta)
    assert len(golden["names"]) == 4
    for name in golden["names"]:
        mat = os.path.join(tmp_path, name + ".mat")
        open(mat, "wb").write(golden[name + "_matrix_bytes"].tobytes())
        out = os.path.join(tmp_path, name + "_sel")
        assert phyloselect.main(["-i", mat, "-o", out, "-f", path] + str(golden[name + "_select_args"]).split()) == 0
        assert open(os.path.join(out, "data_cluster_indexes.dat"), "rb").read() == golden[name + "_indexes"].tobytes(), name
        files = sorted(f for f in os.listdir(out) if f.startswith("data_fasta_"))
        assert files == [str(f) for f in golden[name + "_fasta_names"]], name
        for f in files:
            assert open(os.path.join(out, f), "rb").read() == golden[name + "_" + f].tobytes(), (name, f)


# ---------------------------------------------------------------------------------------------------------------
# The selection kernels against float64 numpy, entry semantics written out once:
#   -0.0 equals +0.0; NaN sorts last whatever its sign; ties go to the smallest column; an argmin picks the first
#   NaN when there is one (np.argmin); sums are compared with math.fsum.
# ---------------------------------------------------------------------------------------------------------------
def ref_order(row, exclude=None):
    """Columns of a row ascending by value, -0.0 == +0.0, NaN (either sign) last, ties by column."""
    row = np.asarray(row, dtype=np.float64)
    nan = np.isnan(row)
    key = np.where(nan, 0.0, row) + 0.0  # -0.0 + 0.0 = +0.0
    order = np.lexsort((np.arange(len(row)), key, nan))
    return order if exclude is None else order[order != exclude]


def ref_first_argmin(x):
    """np.argmin: the first NaN when there is one, else the first of the smallest values."""
    return int(np.argmin(np.asarray(x, dtype=np.float64)))


def same_values(a, b):
    """Equal as values (-0.0 == +0.0), NaN in the same places."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and bool((a[~np.isnan(a)] == b[~np.isnan(b)]).all())


NEG_NAN = np.copysign(np.nan, -1.0)


def value_family(kind, rows, n, k, rng):
    """A float64 (rows, n) block of one value family; `k` places the float32 collisions at the k-th neighbour."""
    if kind == "continuous":
        return rng.random((rows, n))
    if kind == "quantised":
        return np.floor(rng.random((rows, n)) * 8.0) / 8.0  # n / 8 ties per level
    if kind == "f64_close":
        # the k-th neighbour falls inside a run of entries that are all one float32 apart from nothing: 1e-12 steps
        # around 0.5, far below float32's ulp there (6e-8), in random columns and in random value order
        D = 1.0 + rng.random((rows, n))
        m = min(n, k + 2 + k // 2)
        for i in range(rows):
            cols = rng.choice(n, m, replace=False)
            D[i, cols] = 0.5 + 1e-12 * rng.permutation(m)
        return D
    if kind == "signed_zero":
        return rng.choice(np.array([-0.0, 0.0, 0.25, 1.0]), size=(rows, n), p=[0.3, 0.3, 0.2, 0.2])
    if kind == "nan":
        D = rng.random((rows, n))
        D[rng.random((rows, n)) < 0.1] = np.nan
        D[rng.random((rows, n)) < 0.1] = NEG_NAN
        return D
    if kind == "inf":
        D = rng.random((rows, n))
        D[rng.random((rows, n)) < 0.05] = np.inf
        D[rng.random((rows, n)) < 0.05] = -np.inf
        return D
    if kind == "negative":
        return rng.normal(0.0, 1.0, (rows, n))  # KT-style: correlations, negative entries
    raise ValueError(kind)


FAMILIES = ["continuous", "quantised", "f64_close", "signed_zero", "nan", "inf", "negative"]
LAYOUTS = ["contiguous", "ld", "offset", "block_in", "block_out"]


def device_layout(M, layout):
    """The block M on the device as a contiguous tensor, a column slice of a wider matrix (ld > n_cols) or a view
    one element past an allocation (rows not 16-byte aligned); the padding is NaN so that a stray read shows."""
    rows, n = M.shape
    t = torch.from_numpy(np.ascontiguousarray(M)).cuda()
    if layout == "ld":
        W = torch.full((rows, n + 13), float("nan"), dtype=t.dtype, device="cuda")
        W[:, :n] = t
        return W[:, :n]
    if layout == "offset":
        flat = torch.full((rows * n + 2,), float("nan"), dtype=t.dtype, device="cuda")
        flat[1:1 + rows * n] = t.reshape(-1)
        return flat[1:1 + rows * n].view(rows, n)
    return t


def knn_cases():
    """A sample of (n_cols, k, family, layout, dtype): every valid (n_cols, k) pair once, the other axes cycled."""
    cases = []
    for n in (40, 255, 256, 257, 8191, 8192, 8193, 8192 + 127, 30000):
        for k in sorted(set(kk for kk in (1, 2, 3, 255, 256, 257, 1023, 1024, n - 1) if 1 <= kk <= min(1024, n - 1))):
            q = len(cases)
            cases.append((n, k, FAMILIES[q % 7], LAYOUTS[(q // 2) % 5], (np.float32, np.float64)[(q // 3) % 2]))
    return cases


@pytest.mark.parametrize("n,k,family,layout,dtype", knn_cases())
def test_knn_matches_the_reference_order(n, k, family, layout, dtype):
    rng = np.random.default_rng(n * 1031 + k)
    rows = 6
    M = value_family(family, rows, n, k, rng).astype(dtype)
    row0 = {"block_in": n - rows - 1, "block_out": n + 5}.get(layout, 0)
    idx, dist = phyloselect.knn_graph(device_layout(M, layout), k, row0=row0)
    idx, dist = idx.cpu().numpy(), dist.cpu().numpy()
    for i in range(rows):
        want = ref_order(M[i], exclude=row0 + i)[:k]
        assert np.array_equal(idx[i], want), (i, np.nonzero(idx[i] != want)[0][:5])
        assert np.array_equal(dist[i], M[i][want].astype(np.float32), equal_nan=True), i


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_knn_signed_zeros_are_equal(dtype):
    """-0.0 and +0.0 are one value: the tie goes to the smaller column, whichever of the two it holds."""
    D = np.ones((4, 300), dtype=dtype)
    D[:, 7] = -0.0
    D[:, 3] = 0.0
    D[1, 9] = -0.0
    D[2, 3] = -0.0
    D[2, 7] = 0.0
    idx, _ = phyloselect.knn_graph(torch.from_numpy(D).cuda(), 3, row0=100)
    assert idx.cpu().numpy()[:, :2].tolist() == [[3, 7], [3, 7], [3, 7], [3, 7]]
    assert idx.cpu().numpy()[1, 2] == 9


def test_knn_float64_ranks_by_full_precision():
    """float64 entries that round to one float32 are ordered by value, not as ties by column."""
    n, k = 500, 10
    D = 0.5 + 1e-12 * (n - np.arange(n, dtype=np.float64))[None, :].repeat(3, axis=0)
    assert len(np.unique(D[0].astype(np.float32))) == 1
    idx, dist = phyloselect.knn_graph(torch.from_numpy(D).cuda(), k, row0=n)
    assert (idx.cpu().numpy() == np.arange(n - 1, n - 1 - k, -1)[None, :]).all()
    assert (dist.cpu().numpy() == np.float32(0.5)).all()


def test_knn_refuses_k_outside_its_range():
    D = torch.rand((5, 40), device="cuda")
    for k in (0, 1025, 40):
        with pytest.raises(PhyloligoError):
            phyloselect.knn_graph(D, k)
    with pytest.raises(PhyloligoError):
        phyloselect.knn_graph(torch.rand((5, 3000), device="cuda", dtype=torch.float64), 1025)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("family,layout", [("continuous", "ld"), ("signed_zero", "offset"), ("nan", "contiguous"),
                                           ("negative", "ld"), ("f64_close", "offset"), ("inf", "contiguous")])
def test_kth_smallest_matches_the_sorted_row(family, layout, dtype):
    rng = np.random.default_rng(len(family) * 7 + len(layout))
    for n in (1, 257, 8193):
        M = value_family(family, 5, n, max(1, n // 3), rng).astype(dtype)
        Dd = device_layout(M, layout)
        for k in (1, max(1, n // 3), n):
            got = phyloselect.kth_smallest(Dd, k).cpu().numpy()
            assert got.dtype == dtype
            want = np.array([M[i][ref_order(M[i])[k - 1]] for i in range(len(M))], dtype=dtype)
            assert same_values(got, want), (n, k, got, want)


def fsum_close(got, x):
    """got is a float64 sum of x: NaN / inf as the exact sum has them, else within n 2^-53 sum|x| of math.fsum."""
    x = np.asarray(x, dtype=np.float64)
    if not np.isfinite(x).all():
        want = x.sum()  # NaN, or the infinity of the one sign present
        return np.isnan(want) and np.isnan(got) or want == got
    return abs(got - math.fsum(x.tolist())) <= len(x) * 2.0 ** -53 * np.abs(x).sum()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n", [0, 1, 255, 256, 769, 1023, 1024, 1025, 100003])
def test_row_sums_against_fsum(n, dtype):
    """Every tail of the four-accumulator loop; all columns, a rows subset, label masks and ld > n_cols."""
    rng = np.random.default_rng(n + 5)
    rows = 7
    M = (rng.normal(0.0, 1.0, (rows, n)) * 10.0 ** rng.integers(-3, 4, (rows, n))).astype(dtype)
    if n:
        M[2, n // 2] = np.nan
        M[3, n - 1] = np.inf
        M[4, 0] = -np.inf
    for layout in (("contiguous", "ld") if n == 0 else ("contiguous", "ld", "offset")):
        Dd = device_layout(M, layout)
        got = phyloselect.row_sums(Dd).cpu().numpy()
        assert all(fsum_close(got[i], M[i]) for i in range(rows)), layout
        assert np.array_equal(got, phyloselect.row_sums(Dd).cpu().numpy(), equal_nan=True)  # reproducible, bit for bit
        sub = torch.tensor([5, 0, 5, 3], dtype=torch.int64, device="cuda")
        got = phyloselect.row_sums(Dd, rows=sub).cpu().numpy()
        assert all(fsum_close(got[q], M[r]) for q, r in enumerate([5, 0, 5, 3]))
        if n == 0:
            continue
        labels = rng.integers(0, 3, n).astype(np.int32)
        lab = torch.from_numpy(labels).cuda()
        for row_labels in (np.zeros(rows, np.int32), rng.integers(0, 3, rows).astype(np.int32)):
            got = phyloselect.row_sums(Dd, labels=lab, row_labels=torch.from_numpy(row_labels).cuda()).cpu().numpy()
            assert all(fsum_close(got[i], M[i][labels == row_labels[i]]) for i in range(rows))
        # every column matches, and none does (the sum of nothing is 0.0)
        got = phyloselect.row_sums(Dd, labels=torch.zeros(n, dtype=torch.int32, device="cuda"),
                                   row_labels=torch.zeros(rows, dtype=torch.int32, device="cuda")).cpu().numpy()
        assert all(fsum_close(got[i], M[i]) for i in range(rows))
        got = phyloselect.row_sums(Dd, labels=lab, row_labels=torch.full((rows,), 7, dtype=torch.int32, device="cuda"))
        assert (got.cpu().numpy() == 0.0).all()


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("k,n", [(1, 1000), (2, 333), (7, 5000), (64, 1000)])
def test_assign_to_medoids_is_np_argmin(k, n, dtype):
    """Ties (quantised values), +-0, NaN of either sign in any medoid row, a matrix wider than its rows (ld > n)."""
    rng = np.random.default_rng(k * 100 + n)
    M = rng.choice(np.array([-0.0, 0.0, 0.5, 1.0, 2.0]), size=(k + 3, n))
    M[rng.random(M.shape) < 0.05] = np.nan
    M[rng.random(M.shape) < 0.05] = NEG_NAN
    M[:, :4] = np.nan  # a whole column of NaN: the first medoid
    M = M.astype(dtype)
    rows = rng.permutation(k + 3)[:k]
    for layout in ("contiguous", "ld"):
        got = phyloselect.assign_to_medoids(device_layout(M, layout), torch.from_numpy(rows).cuda()).cpu().numpy()
        assert np.array_equal(got, np.argmin(M[rows].astype(np.float64), axis=0)), layout


def test_cluster_argmin_is_the_first_argmin_per_cluster():
    """NaN costs of both signs, +-0, empty clusters, labels outside [0, k), no points at all and k > n."""
    rng = np.random.default_rng(8)
    for n, k in ((1000, 7), (5, 9), (0, 3), (3000, 1)):
        cost = rng.choice(np.array([-0.0, 0.0, 1.0, -2.0, np.inf, -np.inf, 3.5]), size=n)
        if n >= 100:
            cost[rng.random(n) < 0.02] = np.nan
            cost[rng.random(n) < 0.02] = NEG_NAN
        labels = rng.integers(-2, k + 2, n).astype(np.int32)
        if k == 7:
            labels[labels == 3] = 4  # cluster 3 empty
        idx, best, count = phyloselect.cluster_argmin(torch.from_numpy(cost).cuda(), torch.from_numpy(labels).cuda(), k)
        idx, best, count = idx.cpu().numpy(), best.cpu().numpy(), count.cpu().numpy()
        for c in range(k):
            members = np.nonzero(labels == c)[0]
            assert count[c] == len(members), (n, k, c)
            if len(members) == 0:
                assert idx[c] == -1 and best[c] == 0.0, (n, k, c)
                continue
            want = members[ref_first_argmin(cost[members])]
            assert idx[c] == want and same_values(best[c], cost[want]), (n, k, c, idx[c], want)


def bc_matrix_with_empty_contigs(empty, nan_sign):
    """BC distances of real-shaped profiles with the contigs `empty` all-zero: 0/0 = NaN on their diagonal entries
    (and between two of them), with the NaN's sign bit set as given."""
    seqs = synth.make_sequences(200, 3000, seed=9)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs])
    X[list(empty)] = 0.0
    with np.errstate(invalid="ignore", divide="ignore"):
        D = po.pairwise_np(X, "BC")
    D[np.isnan(D)] = np.copysign(np.nan, nan_sign)
    return D


@pytest.mark.parametrize("nan_sign", [1.0, -1.0])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("empty", [(50,), (50, 120)])
def test_kmedoids_with_empty_contigs_keeps_nan_cost_medoids(empty, dtype, nan_sign):
    """An empty contig's cost is NaN: np.argmin picks it, NaN < cost is false and the medoid stays, as the
    reference's _update_medoid_ics_in_place does."""
    D = bc_matrix_with_empty_contigs(empty, nan_sign).astype(dtype)
    assert np.isnan(D[empty[0], empty[0]])
    for k in (2, 3, 5):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            labels, medoids, n_iter = so.kmedoids_fit(D.astype(np.float64), n_clusters=k)
            km = phyloselect.KMedoids(n_clusters=k).fit(D)
        assert np.array_equal(km.medoid_indices_, medoids), (k, km.medoid_indices_, medoids)
        assert np.array_equal(km.labels_, labels) and km.n_iter_ == n_iter, k


def test_command_line_kmedoids_bc_with_an_all_n_record(tmp_path):
    from phyloligo_b200 import phyloligo
    seqs = synth.make_sequences(150, 3000, seed=21)
    seqs[40] = b"N" * 2500
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    out = os.path.join(tmp_path, "out")
    assert phyloselect.main(["--assembly", fasta, "-d", "BC", "-m", "kmedoids", "-k", "3", "-o", out]) == 0
    # the oracle on the matrix the command computed on the device
    res, n, _ = phyloligo._profile_file(fasta, "1111", "both", ("freq32",))
    D = engine.distance_matrix_device(res["freq32"], phyloligo._large_metric("BC"), torch.float32, symmetric=True).cpu().numpy()
    assert np.isnan(D[40, 40])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want, _, _ = so.kmedoids_fit(D.astype(np.float64), n_clusters=3)
    rows = [tuple(int(v) for v in line.split()) for line in open(os.path.join(out, "data_cluster_indexes.dat"))]
    assert rows == sorted((int(c), i) for i, c in enumerate(want))


def test_tsne_affinities_float64_collisions_at_the_neighbour_boundary():
    """The float64 neighbours t-SNE takes are the k smallest by value, where float32 would see a run of ties."""
    from oracle import tsne_oracle as to
    rng = np.random.default_rng(4)
    n, perplexity = 300, 5.0
    k = int(3 * perplexity + 1)
    # every row: k - 4 distinct near neighbours, then a run of 12 entries 1e-12 apart (one float32) across the k-th
    D = 1.0 + rng.random((n, n))
    for i in range(n):
        cols = rng.choice(np.delete(np.arange(n), i), k + 8, replace=False)
        D[i, cols[:k - 4]] = 0.1 + 0.01 * rng.permutation(k - 4)
        D[i, cols[k - 4:]] = 0.5 + 1e-12 * rng.permutation(12)
    np.fill_diagonal(D, 0.0)
    got = phyloselect.tsne_affinities(torch.from_numpy(D).cuda(), perplexity, as_sparse=True)
    want = to.joint_probabilities(D, perplexity)
    assert want.nnz > n * k
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.abs(got.data - want.data).max() <= 1e-9
    # all k neighbours of every row equidistant: the perplexity search drives every P_ij to 0 and P is empty
    for i in range(n):
        D[i, np.argsort(D[i])[1:k + 1]] = 0.5
    got = phyloselect.tsne_affinities(torch.from_numpy(D).cuda(), perplexity, as_sparse=True)
    want = to.joint_probabilities(D, perplexity)
    assert want.nnz == 0 and got.nnz == 0 and np.array_equal(got.indptr, want.indptr)
