"""GPU parity of phyloselect's HDBSCAN (phyloligo_b200/phyloselect.py, csrc/po_hdbscan.cu, po_matrix_kth in
csrc/po_select.cu) against the numpy oracle (oracle/hdbscan_oracle.py) and scikit-learn's HDBSCAN."""
import os

import numpy as np
import pytest
import torch
from sklearn.cluster import HDBSCAN as SkHDBSCAN

from oracle import hdbscan_oracle as ho
from oracle import phylo_oracle as po
from phyloligo_b200 import engine, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError
from test_hdbscan_oracle import assert_same_clustering, blobs, jsd_matrix

pytestmark = pytest.mark.gpu


def quantised(n, seed, levels=6):
    """A tie-heavy matrix: distances rounded to a few levels."""
    D = blobs(n, seed)
    return np.round(D / D.max() * levels) / levels


def kt_style(n, seed):
    """Similarities-like matrix with 1 on the diagonal (as KT), and duplicate rows."""
    rng = np.random.default_rng(seed)
    P = rng.normal(0, 1, size=(n, 5))
    P[n // 2: n // 2 + 10] = P[:10]
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1)) / 4.0
    np.fill_diagonal(D, 1.0)
    return D


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("make,n", [(blobs, 500), (kt_style, 300), (quantised, 400), (jsd_matrix, 250)])
def test_core_distances_are_matrix_entries_bit_for_bit(make, n, dtype):
    D = make(n, 3).astype(dtype)
    Dd = torch.from_numpy(D).cuda()
    for ms in (1, 5, 40, n - 1):
        got = phyloselect.kth_smallest(Dd, ms + 1).cpu().numpy()
        assert got.dtype == dtype
        assert np.array_equal(got.view(np.uint8), np.ascontiguousarray(ho.core_distances(D, ms)).view(np.uint8)), ms


def test_core_distances_keep_float64_precision():
    # entries that round to one float32 must not be confused
    base = np.full((64, 64), 1.0)
    base += np.arange(64)[None, :] * 1e-12
    D = np.minimum(base, base.T)
    got = phyloselect.kth_smallest(torch.from_numpy(D).cuda(), 7).cpu().numpy()
    assert np.array_equal(got, np.partition(D, 6, axis=1)[:, 6])


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("make,n,mcs,ms", [(blobs, 700, 5, None), (quantised, 600, 5, 3), (kt_style, 300, 5, 2),
                                          (jsd_matrix, 800, 15, 3), (blobs, 3000, 40, None)])
def test_mst_labels_and_condensed_tree_equal_the_oracle(make, n, mcs, ms, dtype):
    D = make(n, 5).astype(dtype)
    res = ho.hdbscan(D, mcs, ms)
    h = phyloselect.HDBSCAN(min_cluster_size=mcs, min_samples=ms).fit(D)
    u, v, w = res["mst"]
    mst = h.minimum_spanning_tree_
    assert np.array_equal(mst[:, 0], u) and np.array_equal(mst[:, 1], v) and np.array_equal(mst[:, 2], w.astype(np.float64))
    assert np.array_equal(h.labels_, res["labels"]) and np.array_equal(h.probabilities_, res["probabilities"])
    for f in ("parent", "child", "lambda_val", "child_size"):
        assert np.array_equal(h.condensed_tree_[f], res["condensed_tree"][f]), f
    if make is quantised:
        assert len(np.unique(w)) < 20


@pytest.mark.parametrize("kind,n,seed,mcs,ms", [("blobs", 300, 2, 5, 1), ("blobs", 1000, 3, 5, 1), ("jsd", 1500, 7, 5, 1)])
def test_equals_scikit_learn_on_distinct_weight_sets(kind, n, seed, mcs, ms):
    D = blobs(n, seed) if kind == "blobs" else jsd_matrix(n, seed)
    h = phyloselect.HDBSCAN(min_cluster_size=mcs, min_samples=ms).fit(D)
    w = h.minimum_spanning_tree_[:, 2]
    assert len(np.unique(w)) == len(w)
    msc = ho.clamp_min_samples(n, mcs, ms)
    sk = SkHDBSCAN(min_cluster_size=mcs, min_samples=msc + 1, metric="precomputed", copy=True).fit(D.astype(np.float64))
    assert_same_clustering(h.labels_, h.probabilities_, sk.labels_, sk.probabilities_)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_refusals_name_the_entry(dtype):
    D = blobs(100, 1).astype(dtype)
    A = D.copy()
    A[7, 42] = np.nextafter(A[7, 42], dtype(10))
    with pytest.raises(PhyloligoError, match=r"not symmetric: entry \(7, 42\)"):
        phyloselect.HDBSCAN().fit(A)
    N = D.copy()
    N[63, 12] = N[12, 63] = np.nan
    with pytest.raises(PhyloligoError, match=r"entry \(12, 63\) is NaN"):
        phyloselect.HDBSCAN().fit(N)
    inf = D.copy()
    inf[99, 98] = inf[98, 99] = np.inf
    with pytest.raises(PhyloligoError, match=r"entry \(98, 99\) is infinite"):
        phyloselect.HDBSCAN().fit(inf)
    with pytest.raises(PhyloligoError, match="square"):
        phyloselect.HDBSCAN().fit(D[:, :50])
    with pytest.raises(ValueError, match="min_cluster_size=1"):
        phyloselect.HDBSCAN(min_cluster_size=1).fit(D)


def test_device_tensor_in_place_and_profiles_never_leave_the_device():
    seqs = synth.make_sequences(500, 4000, seed=21)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs]).astype(np.float32)
    Xd = torch.from_numpy(X).cuda()
    Dd = engine.distance_matrix_device(Xd, "JSD", torch.float32, symmetric=True)
    before = Dd.clone()
    a = phyloselect.HDBSCAN(min_cluster_size=5).fit(Dd)
    assert torch.equal(Dd, before)
    b = phyloselect.HDBSCAN(min_cluster_size=5, metric="JSD").fit(Xd)
    c = phyloselect.HDBSCAN(min_cluster_size=5, metric="JSD").fit(X)
    res = ho.hdbscan(Dd.cpu().numpy(), 5)
    for h in (a, b, c):
        assert np.array_equal(h.labels_, res["labels"]) and np.array_equal(h.probabilities_, res["probabilities"])
        assert np.array_equal(h.minimum_spanning_tree_, a.minimum_spanning_tree_)


def _read_dir(path):
    return {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


def test_command_line(tmp_path, capsys):
    seqs = synth.make_sequences(300, 3000, seed=9)
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs])
    D = po.pairwise_np(X, "JSD")
    np.savetxt(os.path.join(tmp_path, "m.txt"), D, delimiter="\t")
    D.astype(np.float32).tofile(os.path.join(tmp_path, "m.bin"))
    from phyloligo_b200 import phyloligo
    res, _, _ = phyloligo._profile_file(fasta, "1111", "both", ("freq32",))
    D_dev = engine.distance_matrix_device(res["freq32"], "JSD", torch.float32, symmetric=True).cpu().numpy()
    cases = (("txt", ["-i", os.path.join(tmp_path, "m.txt")], np.loadtxt(os.path.join(tmp_path, "m.txt"))),
             ("memmap", ["-i", os.path.join(tmp_path, "m.bin"), "--large", "memmap"], D.astype(np.float32)),
             ("device", ["--assembly", fasta, "-d", "JSD", "--pattern", "1111"], D_dev))
    for tag, args, M in cases:
        labels = ho.hdbscan(M, 5, 2)["labels"]
        assert (labels == -1).any() and labels.max() >= 1, tag
        want = os.path.join(tmp_path, "want_" + tag)
        os.makedirs(want)
        phyloselect.write_cluster_indexes(labels, os.path.join(want, "data_cluster_indexes.dat"))
        phyloselect.write_fastafile(labels, fasta, want)
        capsys.readouterr()
        out = os.path.join(tmp_path, "hdb_" + tag)
        assert phyloselect.main(args + ["-m", "hdbscan", "--minclustersize", "5", "--minsamples", "2", "-o", out, "-f", fasta]) == 0
        hdb_lines = capsys.readouterr().out.replace(out, "OUT").splitlines()
        got = _read_dir(out)
        assert got == _read_dir(want), tag
        assert "data_fasta_unclust.fa" in got
        km = os.path.join(tmp_path, "km_" + tag)
        assert phyloselect.main(args + ["-m", "kmedoids", "-k", "3", "-o", km, "-f", fasta]) == 0
        assert capsys.readouterr().out.replace(km, "OUT").splitlines() == hdb_lines, tag


def test_twenty_thousand_device_profiled_contigs():
    dev = engine.require_cuda()
    text, b, e, _ = synth.device_fasta(20000, 3000, 17, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    Dd = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    h = phyloselect.HDBSCAN(min_cluster_size=5).fit(Dd)
    D = Dd.cpu().numpy()
    del Dd
    core = ho.core_distances(D, 5)
    u, v, w = ho.mst_prim_streaming(D, core)
    mst = h.minimum_spanning_tree_
    assert np.array_equal(mst[:, 0], u) and np.array_equal(mst[:, 1], v) and np.array_equal(mst[:, 2], w.astype(np.float64))
    labels, probs, _, _, _ = phyloselect.hdbscan_tree(u, v, w.astype(np.float64), 20000, 5)
    assert np.array_equal(h.labels_, labels) and np.array_equal(h.probabilities_, probs)
    assert labels.max() >= 1
