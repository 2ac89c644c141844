"""phyloselect past device memory: row panels of the distance matrix (phyloligo_b200/panels.py, DESIGN.md 4.12).

Every panel of a ProfileSource must be bit for bit the rows of the resident matrix, every consumer (neighbour graph,
t-SNE, HDBSCAN, K-medoids) must give on panels exactly what it gives on the resident matrix, with the same refusals,
and the command line must write the same files when the matrix does not fit.
"""
import os
import warnings

import numpy as np
import pytest
import torch

from phyloligo_b200 import engine, io_formats, panels, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError, TILE

pytestmark = pytest.mark.gpu

METRICS = ["Eucl", "EuclGram", "JSD", "KT", "BC", "SC"]


def profiles(n, dim=256, seed=0):
    """Normalised float32 profiles with an all-zero row and a constant row (SC: NaN, KT: 0) when n allows."""
    rng = np.random.default_rng(seed)
    X = rng.gamma(0.7, 1.0, (n, dim))
    X[rng.random((n, dim)) < 0.05] = 0.0
    X /= np.maximum(X.sum(axis=1, keepdims=True), 1e-300)
    if n > 3:
        X[n // 3] = 0.0
        X[(2 * n) // 3] = 1.0 / dim
    return torch.from_numpy(X.astype(np.float32)).cuda()


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def heights(n):
    return [TILE, 3 * TILE, -(-n // TILE) * TILE]


@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 1000, 2049])
@pytest.mark.parametrize("metric", METRICS)
def test_profile_panels_equal_resident_rows(metric, n):
    X = profiles(n, seed=n)
    want = engine.distance_matrix_device(X, metric, torch.float32, symmetric=True)
    for h in heights(n):
        src = panels.ProfileSource(X, metric, panel_rows=h)
        spans = []
        for r0, r1, P in src.panels():
            assert same_bits(P, want[r0:r1]), (metric, n, h, r0)
            spans.append((r0, r1))
        assert spans[0][0] == 0 and spans[-1][1] == n and all(b[0] == a[1] for a, b in zip(spans, spans[1:]))
        assert all((r1 - r0) == h for r0, r1 in spans[:-1])
        idx = torch.tensor([n - 1, 0, n // 2, n - 1], device="cuda")
        assert same_bits(src.rows(idx), want[idx])


@pytest.mark.parametrize("n", [2, 129, 1000])
def test_kt_of_one_dimension(n):
    X = profiles(n, dim=1, seed=3)
    want = engine.distance_matrix_device(X, "KT", torch.float32, symmetric=True)
    for r0, r1, P in panels.ProfileSource(X, "KT", panel_rows=TILE).panels():
        assert same_bits(P, want[r0:r1])


def write_memmap(D, path):
    D.cpu().numpy().astype(np.float32).tofile(path)
    return panels.FileSource(path, D.shape[0], panel_rows=2 * TILE)


@pytest.mark.parametrize("fmt", ["memmap", "h5py"])
def test_file_source_rows(tmp_path, fmt):
    n = 1000
    A = np.random.default_rng(1).random((n, n), dtype=np.float32)
    path = str(tmp_path / "m.bin")
    if fmt == "memmap":
        A.tofile(path)
        ref = np.memmap(path, dtype=np.float32, mode="r", shape=(n, n))
    else:
        io_formats.write_hdf5(path, "distances", A)
        ref = io_formats.read_hdf5(path, "distances")
    n2, offset, dtype = panels.file_matrix(path, fmt)
    src = panels.FileSource(path, n2, offset=offset, dtype=dtype, panel_rows=3 * TILE)
    seen = 0
    for r0, r1, P in src.panels():
        assert np.array_equal(P.cpu().numpy(), ref[r0:r1])
        seen = r1
    assert seen == n and n % (3 * TILE) != 0
    idx = torch.tensor([999, 3, 3, 500, 0])
    assert np.array_equal(src.rows(idx).cpu().numpy(), ref[idx.numpy()])
    assert np.array_equal(src.column_strip(384, 768).cpu().numpy(), ref[:, 384:768])
    src.close()


N_FIT = 2500


@pytest.fixture(scope="module")
def fit_case(tmp_path_factory):
    X = profiles(N_FIT, seed=11)
    # a few tight groups so that HDBSCAN and K-medoids find structure
    centres = profiles(6, seed=12)
    X[: N_FIT // 2] = 0.7 * X[: N_FIT // 2] + 0.3 * centres[torch.arange(N_FIT // 2, device="cuda") % 6]
    D = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    path = str(tmp_path_factory.mktemp("panels") / "jsd.memmap")
    D.cpu().numpy().tofile(path)
    return X, D, path


def sources(fit_case):
    X, D, path = fit_case
    yield "profiles", panels.ProfileSource(X, "JSD", panel_rows=3 * TILE)
    yield "file", panels.FileSource(path, N_FIT, panel_rows=5 * TILE)


def test_knn_graph_on_panels(fit_case):
    _, D, _ = fit_case
    want_i, want_d = phyloselect.knn_graph(D, 15)
    for name, src in sources(fit_case):
        i, d = phyloselect.knn_graph(src, 15)
        assert torch.equal(i, want_i) and same_bits(d, want_d), name


@pytest.mark.parametrize("max_iter", [250, 300])
def test_tsne_on_panels(fit_case, max_iter):
    _, D, _ = fit_case
    want = phyloselect.TSNE(perplexity=30.0, early_exaggeration=12.0, max_iter=max_iter, random_state=0).fit(D)
    for name, src in sources(fit_case):
        got = phyloselect.TSNE(perplexity=30.0, early_exaggeration=12.0, max_iter=max_iter, random_state=0).fit(src)
        assert np.array_equal(got.embedding_, want.embedding_), name
        assert got.kl_divergence_ == want.kl_divergence_ and got.n_iter_ == want.n_iter_, name


@pytest.mark.parametrize("mcs", [5, 50])
def test_hdbscan_on_panels(fit_case, mcs):
    _, D, _ = fit_case
    want = phyloselect.HDBSCAN(min_cluster_size=mcs).fit(D)
    for name, src in sources(fit_case):
        got = phyloselect.HDBSCAN(min_cluster_size=mcs).fit(src)
        assert np.array_equal(got.labels_, want.labels_), name
        assert np.array_equal(got.probabilities_, want.probabilities_), name
        assert np.array_equal(got.condensed_tree_, want.condensed_tree_), name
        assert np.array_equal(got.single_linkage_tree_, want.single_linkage_tree_), name
        assert np.array_equal(got.minimum_spanning_tree_, want.minimum_spanning_tree_), name


@pytest.mark.parametrize("init", ["heuristic", "random"])
def test_kmedoids_on_panels(fit_case, init):
    _, D, _ = fit_case

    def fit(X):
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            km = phyloselect.KMedoids(n_clusters=40, init=init, random_state=5).fit(X)
        return km, [str(w.message) for w in caught]

    want, want_warn = fit(D)
    for name, src in sources(fit_case):
        got, got_warn = fit(src)
        assert np.array_equal(got.labels_, want.labels_) and np.array_equal(got.medoid_indices_, want.medoid_indices_), name
        assert got.n_iter_ == want.n_iter_ and got_warn == want_warn, name
        assert np.array_equal(got.cluster_centers_, D[torch.from_numpy(want.medoid_indices_).cuda()].cpu().numpy()), name


def refusal(fn):
    with pytest.raises(PhyloligoError) as e:
        fn()
    return str(e.value)


def test_refusals_name_the_resident_entry(tmp_path):
    n = 700
    D = engine.distance_matrix_device(profiles(n, seed=4), "JSD", torch.float32, symmetric=True)
    cases = []
    E = D.clone()
    E[300, 310] = E[310, 300] = float("nan")  # NaN in the second panel, both entries
    cases.append(("nan", E, ("hdbscan", "tsne")))
    E = D.clone()
    E[2 * TILE, 5] = -1e-3  # negative at the second panel's first row
    cases.append(("negative", E, ("tsne",)))
    E = D.clone()
    E[400, 20] = E[400, 20] * 1.5  # asymmetry off the first panel's diagonal square
    cases.append(("asymmetric", E, ("hdbscan",)))
    for what, E, methods in cases:
        path = str(tmp_path / (what + ".bin"))
        for method in methods:
            fit = (lambda X: phyloselect.HDBSCAN().fit(X)) if method == "hdbscan" else (
                lambda X: phyloselect.TSNE(perplexity=5.0, random_state=0).fit(X))
            want = refusal(lambda: fit(E))
            got = refusal(lambda: fit(write_memmap(E, path)))
            assert got == want, (what, method, got, want)
    # a profile source checks the same entries (a NaN row of SC: constant profile)
    X = profiles(n, seed=4)
    want = refusal(lambda: phyloselect.HDBSCAN().fit(engine.distance_matrix_device(X, "SC", torch.float32, symmetric=True)))
    assert refusal(lambda: phyloselect.HDBSCAN().fit(panels.ProfileSource(X, "SC", panel_rows=TILE))) == want


def squeeze_budget(monkeypatch, n):
    """A budget that holds the working state and a few panels of n rows, but not the n x n matrix."""
    budget = panels.state_bytes(n) + 2 * 3 * TILE * n * 4 + 4096
    assert not panels.fits(n, 4, budget) and panels.panel_rows_for(n, 4, budget) == 3 * TILE
    monkeypatch.setattr(panels, "device_budget", lambda device=None: budget)


@pytest.fixture(scope="module")
def assembly(tmp_path_factory):
    d = tmp_path_factory.mktemp("asm")
    fa = str(d / "asm.fa")
    synth.write_fasta(fa, synth.make_sequences(1100, 1500, seed=9))
    return fa


def run_cli(args, out):
    assert phyloselect.main(args + ["-o", out]) == 0
    return {f: open(os.path.join(out, f), "rb").read() for f in sorted(os.listdir(out))}


@pytest.mark.parametrize("method", ["hdbscan", "kmedoids"])
def test_command_line_past_the_device(tmp_path, monkeypatch, assembly, method):
    n = 1100
    extra = ["-m", method] + (["-k", "6"] if method == "kmedoids" else []) + ["-p", "30"]
    want = run_cli(["--assembly", assembly, "--tsne-out", str(tmp_path / "r" / "tsne.txt")] + extra, str(tmp_path / "r"))
    # the same matrix as a phyloligo.py --large memmap file
    from phyloligo_b200 import phyloligo
    res, _, _ = phyloligo._profile_file(assembly, "1111", "both", ("freq32",))
    mm = str(tmp_path / "m.memmap")
    engine.distance_matrix_device(res["freq32"], "JSD", torch.float32, symmetric=True).cpu().numpy().tofile(mm)
    squeeze_budget(monkeypatch, n)
    got = run_cli(["--assembly", assembly, "--tsne-out", str(tmp_path / "p" / "tsne.txt")] + extra, str(tmp_path / "p"))
    assert got == want
    got = run_cli(["-i", mm, "--large", "memmap", "-f", assembly, "--tsne-out", str(tmp_path / "f" / "tsne.txt")] + extra,
                  str(tmp_path / "f"))
    assert got == want
    assert any(f.startswith("data_fasta_") for f in want) and "data_cluster_indexes.dat" in want


def test_command_line_refuses_trees_past_the_device(tmp_path, monkeypatch, assembly):
    squeeze_budget(monkeypatch, 1100)
    for args, what in ((["-m", "hclust", "-k", "4"], "-m hclust"), (["-m", "hdbscan", "--tree-out", str(tmp_path / "t.nwk")], "--tree-out"),
                       (["-m", "hdbscan", "--tree-out", str(tmp_path / "t.nwk"), "--tree-method", "nj"], "--tree-out")):
        with pytest.raises(PhyloligoError, match=r"%s of 1100 rows needs \d+ bytes of device memory" % what):
            phyloselect.main(["--assembly", assembly, "-o", str(tmp_path / "o")] + args)
        assert not os.path.exists(str(tmp_path / "o" / "data_cluster_indexes.dat"))


def test_one_run_past_the_device():
    """n such that the float32 matrix (4 n^2 bytes) exceeds the device's memory: the automatic choice takes
    panels; the neighbour graph and an HDBSCAN fit complete, and the neighbours of 64 sampled rows agree with a
    float64 evaluation of the same JSD formula."""
    total = torch.cuda.get_device_properties(0).total_memory
    n = int(np.sqrt(total / 4)) // 1000 * 1000 + 10000
    X = profiles(n, dim=256, seed=21)
    src = panels.profile_source(X, "JSD")
    assert not src.resident and 4 * n * n > total
    k = 10
    idx, dist = phyloselect.knn_graph(src, k)
    rows = torch.from_numpy(np.random.default_rng(0).choice(n, 64, replace=False)).cuda()
    A = X[rows].double()
    ref = torch.empty((64, n), dtype=torch.float64, device="cuda")
    for c0 in range(0, n, 4096):
        B = X[c0:c0 + 4096].double()
        H = 0.5 * (A[:, None, :] + B[None, :, :])
        d1 = A[:, None, :] * torch.log(A[:, None, :] / H)
        d2 = B[None, :, :] * torch.log(B[None, :, :] / H)
        ref[:, c0:c0 + 4096] = 0.5 * (torch.nan_to_num(d1, nan=0.0, posinf=0.0, neginf=0.0).sum(2)
                                      + torch.nan_to_num(d2, nan=0.0, posinf=0.0, neginf=0.0).sum(2))
    ref[torch.arange(64), rows] = float("inf")  # a row's own column is not a neighbour
    got = ref.gather(1, idx[rows].long())
    assert torch.allclose(dist[rows].double(), got, rtol=1e-6, atol=1e-12)
    kbest = torch.topk(ref, k, largest=False).values
    assert torch.allclose(got, kbest, rtol=1e-6, atol=1e-12)  # the same neighbours but for exact ties
    hd = phyloselect.HDBSCAN(min_cluster_size=5).fit(src)
    assert hd.labels_.shape == (n,) and hd.minimum_spanning_tree_.shape == (n - 1, 3)
