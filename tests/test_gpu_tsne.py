"""GPU parity of phyloselect's t-SNE (phyloligo_b200/phyloselect.py, csrc/po_tsne.cu) against the numpy oracle
(oracle/tsne_oracle.py) and scikit-learn's TSNE(metric="precomputed", angle=0.0)."""
import os

import numpy as np
import pytest
import torch
from sklearn.manifold import TSNE as SkTSNE
from sklearn.manifold import trustworthiness
from sklearn.utils import check_random_state

from oracle import phylo_oracle as po
from oracle import tsne_oracle as to
from phyloligo_b200 import engine, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError
from test_hdbscan_oracle import blobs, jsd_matrix
from test_tsne_oracle import sklearn_gradient, sklearn_P

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("perplexity", [5.0, 30.0, 100.0])
@pytest.mark.parametrize("n", [300, 1000, 2500])
def test_affinities_equal_scikit_learn_and_the_oracle(n, perplexity, dtype):
    D = blobs(n, 11).astype(dtype)  # distinct distances: scikit-learn orders exact ties its own way
    got = phyloselect.tsne_affinities(torch.from_numpy(D).cuda(), perplexity, as_sparse=True)
    for want in (sklearn_P(D, perplexity), to.joint_probabilities(D, perplexity)):
        assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
        assert np.abs(got.data - want.data).max() <= 1e-9
    if n == 300 and perplexity == 100.0:
        assert got.nnz == n * (n - 1)  # k = n - 1: every pair


def test_affinities_of_a_jsd_matrix():
    D = jsd_matrix(800, 5)
    got = phyloselect.tsne_affinities(D, 30.0, as_sparse=True)
    want = sklearn_P(D, 30.0)
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.abs(got.data - want.data).max() <= 1e-9


@pytest.mark.parametrize("kind,n", [("blobs", 500), ("jsd", 500), ("blobs", 3000)])
def test_gradient_at_random_and_converged_positions(kind, n):
    D = blobs(n, 4) if kind == "blobs" else jsd_matrix(n, 4)
    P = phyloselect.tsne_affinities(D, 30.0, as_sparse=True)
    converged = phyloselect.TSNE(random_state=1).fit(D).embedding_
    random = np.random.default_rng(n).normal(0, 3, size=(n, 2)).astype(np.float32)
    for Y in (random, converged):
        for ex in (1.0, 12.0):
            g, kl = phyloselect.tsne_gradient(P, Y, exaggeration=ex)
            g_or, kl_or = to.gradient(P, Y, ex)
            g_sk, kl_sk = sklearn_gradient(P, Y, ex)
            assert g.dtype == np.float32
            # 1e-5 of max|g|, except where scikit-learn's own float32 gradient is further from the exact one: near
            # convergence attraction and repulsion cancel to within 1e-4 .. 1e-6 of either, below float32 resolution
            tol = max(1e-5 * np.abs(g_or).max(), np.abs(g_sk - g_or).max())
            assert np.abs(g - g_or).max() <= tol
            assert np.abs(g - g_sk).max() <= 2 * tol
            assert abs(kl - kl_or) <= 1e-5 * abs(kl_or)
            assert abs(kl - kl_sk) <= 3e-4 * abs(kl_sk)  # scikit-learn's KL is a float32 sum


@pytest.mark.parametrize("kind,n,seed", [("blobs", 600, 1), ("jsd", 800, 3), ("blobs", 1200, 2)])
def test_full_fit_matches_scikit_learn(kind, n, seed):
    D = blobs(n, seed) if kind == "blobs" else jsd_matrix(n, seed)
    sk = SkTSNE(metric="precomputed", init="random", random_state=0, angle=0.0).fit(np.array(D))
    t = phyloselect.TSNE(metric="precomputed", init="random", random_state=0, angle=0.0).fit(D)
    assert t.embedding_.dtype == np.float32 and t.embedding_.shape == (n, 2)
    assert t.learning_rate_ == sk.learning_rate_
    assert abs(t.kl_divergence_ - sk.kl_divergence_) <= 0.02 * sk.kl_divergence_
    t_sk = trustworthiness(D, sk.embedding_, n_neighbors=10, metric="precomputed")
    t_dev = trustworthiness(D, t.embedding_, n_neighbors=10, metric="precomputed")
    assert abs(t_sk - t_dev) <= 0.01


def test_random_init_equals_scikit_learns_array_and_fits_are_deterministic():
    D = blobs(700, 6)
    Dd = torch.from_numpy(D).cuda()
    before = Dd.clone()
    for seed in (0, 5):
        a = phyloselect.TSNE(random_state=seed).fit(Dd)
        init = 1e-4 * check_random_state(seed).standard_normal(size=(700, 2)).astype(np.float32)
        b = phyloselect.TSNE(init=init).fit(D)
        assert np.array_equal(a.embedding_, b.embedding_) and a.kl_divergence_ == b.kl_divergence_ and a.n_iter_ == b.n_iter_
    c = phyloselect.TSNE(random_state=5).fit(Dd)
    assert np.array_equal(a.embedding_, c.embedding_) and a.kl_divergence_ == c.kl_divergence_
    assert torch.equal(Dd, before)
    lr = phyloselect.TSNE(random_state=0, learning_rate=200.0, max_iter=300).fit(D)  # float32 update arithmetic
    assert lr.learning_rate_ == 200.0 and np.isfinite(lr.embedding_).all()


def test_profiles_with_a_metric_equal_the_precomputed_matrix():
    seqs = synth.make_sequences(400, 4000, seed=21)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs]).astype(np.float32)
    Xd = torch.from_numpy(X).cuda()
    Dd = engine.distance_matrix_device(Xd, "JSD", torch.float32, symmetric=True)
    want = phyloselect.TSNE(random_state=0).fit(Dd).embedding_
    for src in (Xd, X):
        assert np.array_equal(phyloselect.TSNE(metric="JSD", random_state=0).fit(src).embedding_, want)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_refusals(dtype):
    D = blobs(100, 1).astype(dtype)
    for value, word, (i, j) in ((np.nan, "NaN", (12, 63)), (np.inf, "infinite", (98, 99)), (-1e-3, "negative", (7, 42))):
        A = D.copy()
        A[i, j] = value
        A[j, i] = value
        with pytest.raises(PhyloligoError, match=r"entry \(%d, %d\) is %s" % (i, j, word)):
            phyloselect.TSNE().fit(A)
    Z = D.copy()
    Z[3, 4] = -0.0  # not negative, as in scikit-learn
    phyloselect.TSNE(max_iter=250).fit(Z)
    with pytest.raises(ValueError, match=r"perplexity \(100\.0\) must be less than n_samples \(100\)"):
        phyloselect.TSNE(perplexity=100.0).fit(D)
    with pytest.raises(ValueError, match="at most 1024"):
        phyloselect.TSNE(perplexity=342.0).fit(blobs(1100, 1))
    with pytest.raises(PhyloligoError, match="square"):
        phyloselect.TSNE().fit(D[:, :50])
    with pytest.raises(ValueError, match=r"\(100, 2\) is expected"):
        phyloselect.TSNE(init=np.zeros((99, 2), np.float32)).fit(D)


def test_twenty_thousand_device_profiled_contigs():
    dev = engine.require_cuda()
    text, b, e, _ = synth.device_fasta(20000, 3000, 17, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    Dd = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    P = phyloselect.tsne_affinities(Dd, 30.0, as_sparse=True)
    Y = np.random.default_rng(3).normal(0, 10, size=(20000, 2)).astype(np.float32)
    g, kl = phyloselect.tsne_gradient(P, Y)
    g_or, kl_or = to.gradient(P, Y, chunk=256)
    assert np.abs(g - g_or).max() <= 1e-5 * np.abs(g_or).max()
    assert abs(kl - kl_or) <= 1e-5 * abs(kl_or)
    t = phyloselect.TSNE(random_state=0).fit(Dd)
    assert np.isfinite(t.embedding_).all() and t.n_iter_ >= 250 and np.isfinite(t.kl_divergence_)


def _read_dir(path):
    return {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


def test_command_line(tmp_path):
    seqs = synth.make_sequences(300, 3000, seed=9)
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    X = np.vstack([po.frequency_np(s, "1111", "both") for s in seqs])
    D = po.pairwise_np(X, "JSD")
    np.savetxt(os.path.join(tmp_path, "m.txt"), D, delimiter="\t")
    D.astype(np.float32).tofile(os.path.join(tmp_path, "m.bin"))
    from phyloligo_b200 import phyloligo
    res, _, _ = phyloligo._profile_file(fasta, "1111", "both", ("freq32",))
    D_dev = engine.distance_matrix_device(res["freq32"], "JSD", torch.float32, symmetric=True)
    cases = (("txt", ["-i", os.path.join(tmp_path, "m.txt")], np.loadtxt(os.path.join(tmp_path, "m.txt")), []),
             ("memmap", ["-i", os.path.join(tmp_path, "m.bin"), "--large", "memmap"], D.astype(np.float32), ["-p", "30"]),
             ("device", ["--assembly", fasta, "-d", "JSD", "--pattern", "1111"], D_dev, []))
    for tag, args, M, perp in cases:
        p = float(perp[1]) if perp else 100.0
        want = os.path.join(tmp_path, "want_" + tag + ".tsv")
        np.savetxt(want, phyloselect.TSNE(perplexity=p, random_state=0).fit(M).embedding_, delimiter="\t")
        plain = os.path.join(tmp_path, "plain_" + tag)
        assert phyloselect.main(args + ["-m", "kmedoids", "-k", "3", "-o", plain, "-f", fasta]) == 0
        out = os.path.join(tmp_path, "tsne_" + tag)
        emb = os.path.join(tmp_path, "emb_" + tag + ".tsv")
        assert phyloselect.main(args + perp + ["-m", "kmedoids", "-k", "3", "-o", out, "-f", fasta, "--tsne-out", emb]) == 0
        assert open(emb, "rb").read() == open(want, "rb").read(), tag
        assert _read_dir(out) == _read_dir(plain), tag
        assert len(open(emb).read().splitlines()) == len(seqs)
