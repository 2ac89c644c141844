"""GPU parity of phyloselect's hierarchical clustering (phyloligo_b200/phyloselect.py: linkage, HClust,
--tree-out; csrc/po_linkage.cu) against scipy.cluster.hierarchy.linkage, bit for bit."""
import os

import numpy as np
import pytest
import torch
from scipy.cluster.hierarchy import fcluster
from scipy.cluster.hierarchy import linkage as scipy_linkage
from scipy.spatial.distance import squareform

from oracle import phylo_oracle as po
from phyloligo_b200 import _lib, engine, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError
from test_hdbscan_oracle import blobs, jsd_matrix

pytestmark = pytest.mark.gpu

METHODS = list(phyloselect.LINKAGE_METHODS)


def quantised(n, seed, levels=6):
    D = blobs(n, seed)
    return np.round(D / D.max() * levels) / levels


def kt_style(n, seed):
    """KT-like: negative entries, duplicate rows."""
    rng = np.random.default_rng(seed)
    P = rng.normal(0, 1, size=(n, 5))
    P[n // 2: n // 2 + 10] = P[:10]
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1)) / 4.0 - 0.5
    np.fill_diagonal(D, 0.0)
    return D


def reference(D, method):
    return scipy_linkage(squareform(D, checks=False), method)


def not_a_tree(Z):
    """scipy's result after an all-NaN scan (ward on non-Euclidean data), where its nn_chain reuses a stale index:
    a cluster merged with itself, or a root that does not hold every point."""
    return bool((Z[:, 0] == Z[:, 1]).any() or Z[-1, 3] != len(Z) + 1)


def assert_same(D, method):
    want = reference(D, method)
    if not_a_tree(want):
        with pytest.raises(PhyloligoError, match="NaN"):
            phyloselect.linkage(D, method)
        return
    got = phyloselect.linkage(D, method)
    assert np.array_equal(got, want, equal_nan=True)


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("make,n", [(blobs, 3000), (quantised, 1200), (kt_style, 800), (jsd_matrix, 600)])
def test_equals_scipy_bit_for_bit(make, n, dtype, method):
    D = make(n, 5).astype(dtype)
    assert_same(D, method)


@pytest.mark.parametrize("method", METHODS)
def test_equals_scipy_at_eight_thousand_rows(method):
    D = quantised(8000, 2, levels=40).astype(np.float32)
    assert_same(D, method)


@pytest.mark.parametrize("n,seed", [(30, 17), (30, 23), (30, 28), (60, 1), (60, 4), (60, 8), (60, 18), (120, 3), (120, 13),
                                    (120, 15), (120, 26)])
def test_ward_nan_heights_after_an_all_nan_scan(n, seed):
    # ward on non-Euclidean data: after a merge empties the chain, every distance from the new tip is NaN and
    # scipy pushes its stale y, the slot of the merged cluster; the result is a tree with NaN heights
    D = kt_style(n, seed)
    want = reference(D, "ward")
    assert np.isnan(want[:, 2]).any() and not not_a_tree(want)
    assert np.array_equal(phyloselect.linkage(D, "ward"), want, equal_nan=True)


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("n", [2, 3, 5])
def test_tiny_matrices(n, method):
    for D in (blobs(n, 1), np.zeros((n, n))):
        assert_same(D, method)


def test_device_input_unchanged_and_runs_repeat():
    Dd = torch.from_numpy(jsd_matrix(700, 3)).cuda()
    before = Dd.clone()
    for method in METHODS:
        a = phyloselect.linkage(Dd, method)
        b = phyloselect.linkage(Dd, method)
        assert torch.equal(Dd.view(torch.int32), before.view(torch.int32))
        assert np.array_equal(a.view(np.uint64), b.view(np.uint64)), method


def test_phase_count_is_within_the_bound():
    Dd = torch.from_numpy(blobs(2000, 4)).cuda()
    n = 2000
    for method in METHODS:
        _, _, _, phases = phyloselect.linkage_raw(Dd, method)
        # scans + merges for the NN-chain (at most 3 (n - 1) scans), n - 1 steps for Prim
        assert (phases == n - 1) if method == "single" else (2 * (n - 1) <= phases <= 4 * (n - 1)), (method, phases)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_refusals(dtype, monkeypatch):
    D = blobs(100, 1).astype(dtype)
    A = D.copy()
    A[7, 42] = np.nextafter(A[7, 42], dtype(10))
    with pytest.raises(PhyloligoError, match=r"not symmetric: entry \(7, 42\)"):
        phyloselect.linkage(A)
    N = D.copy()
    N[63, 12] = N[12, 63] = np.nan
    with pytest.raises(PhyloligoError, match=r"entry \(12, 63\) is NaN"):
        phyloselect.linkage(N, "single")
    inf = D.copy()
    inf[99, 98] = inf[98, 99] = np.inf
    with pytest.raises(PhyloligoError, match=r"entry \(98, 99\) is infinite"):
        phyloselect.linkage(inf, "ward")
    for method in ("centroid", "median"):
        with pytest.raises(ValueError, match="not supported"):
            phyloselect.linkage(D, method)
    with pytest.raises(ValueError, match="at least 2"):
        phyloselect.linkage(D[:1, :1])
    with pytest.raises(PhyloligoError, match="square"):
        phyloselect.linkage(D[:, :50])
    # a working copy that does not fit is refused before anything is allocated
    allocated = torch.cuda.memory_allocated()
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1 << 16, 1 << 40))
    memory_allocated = torch.cuda.memory_allocated
    monkeypatch.setattr(torch.cuda, "memory_reserved", lambda device=None: memory_allocated(device))  # no cached blocks
    with pytest.raises(PhyloligoError, match=r"needs %d bytes" % phyloselect.linkage_bytes(100, "average")):
        phyloselect.linkage(torch.from_numpy(D).cuda(), "average")
    assert torch.cuda.memory_allocated() <= allocated + D.nbytes + 4096


def test_hclust_on_profiles_and_on_the_matrix():
    seqs = synth.make_sequences(400, 4000, seed=21)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs]).astype(np.float32)
    Xd = torch.from_numpy(X).cuda()
    Dd = engine.distance_matrix_device(Xd, "JSD", torch.float32, symmetric=True)
    Z = reference(Dd.cpu().numpy(), "average")
    labels = fcluster(Z, 4, "maxclust") - 1
    for h in (phyloselect.HClust(n_clusters=4).fit(Dd), phyloselect.HClust(n_clusters=4, metric="JSD").fit(Xd),
              phyloselect.HClust(n_clusters=4, metric="JSD").fit(X)):
        assert np.array_equal(h.linkage_, Z) and np.array_equal(h.labels_, labels)
    assert labels.min() == 0 and labels.max() == 3


def test_grid_barrier_microbench():
    us = _lib.microbench(4)
    assert 0.0 < us < 100.0


def _read_dir(path):
    return {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


def test_command_line(tmp_path, capsys):
    seqs = synth.make_sequences(300, 3000, seed=9)
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    from phyloligo_b200 import phyloligo
    res, _, _ = phyloligo._profile_file(fasta, "1111", "both", ("freq32",))
    D_dev = engine.distance_matrix_device(res["freq32"], "JSD", torch.float32, symmetric=True).cpu().numpy()
    ids = phyloselect.fasta_record_ids(fasta)
    assert len(ids) == 300 and len(set(ids)) == 300
    for method in ("average", "ward", "single"):
        Z = reference(D_dev, method)
        labels = fcluster(Z, 3, "maxclust") - 1
        want = os.path.join(tmp_path, "want_" + method)
        os.makedirs(want)
        phyloselect.write_cluster_indexes(labels, os.path.join(want, "data_cluster_indexes.dat"))
        phyloselect.write_fastafile(labels, fasta, want)
        phyloselect.write_newick(Z, ids, os.path.join(tmp_path, "want_%s.nwk" % method))
        out = os.path.join(tmp_path, "hc_" + method)
        tree = os.path.join(tmp_path, "got_%s.nwk" % method)
        assert phyloselect.main(["--assembly", fasta, "-d", "JSD", "--pattern", "1111", "-m", "hclust", "-k", "3",
                                 "--linkage", method, "-o", out, "--tree-out", tree]) == 0
        assert _read_dir(out) == _read_dir(want), method
        assert open(tree, "rb").read() == open(os.path.join(tmp_path, "want_%s.nwk" % method), "rb").read()
    # --tree-out with another method, leaves named by row index without -f
    np.savetxt(os.path.join(tmp_path, "m.txt"), D_dev.astype(np.float64), delimiter="\t")
    M = np.loadtxt(os.path.join(tmp_path, "m.txt"))
    out = os.path.join(tmp_path, "km")
    tree = os.path.join(tmp_path, "km.nwk")
    assert phyloselect.main(["-i", os.path.join(tmp_path, "m.txt"), "-m", "kmedoids", "-k", "3", "-o", out, "--tree-out", tree]) == 0
    phyloselect.write_newick(reference(M, "average"), [str(i) for i in range(300)], os.path.join(tmp_path, "want_km.nwk"))
    assert open(tree, "rb").read() == open(os.path.join(tmp_path, "want_km.nwk"), "rb").read()
    capsys.readouterr()
