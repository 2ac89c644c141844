"""Hierarchical clustering without a GPU: the numpy oracle (oracle/linkage_oracle.py) against
scipy.cluster.hierarchy.linkage bit for bit, the library's host stage (po_linkage_tree: stable sort and label) on
the oracle's raw merges, the Newick writer and the size test that refuses a working copy that does not fit."""
import numpy as np
import pytest
from scipy.cluster.hierarchy import cophenet
from scipy.cluster.hierarchy import linkage as scipy_linkage
from scipy.spatial.distance import squareform

from oracle import linkage_oracle as lo
from phyloligo_b200 import phyloselect
from phyloligo_b200._lib import PhyloligoError


def symmetric(A):
    D = np.triu(A, 1)
    return D + D.T


def make(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "ties":  # a few integer levels: heavy ties everywhere
        return symmetric(rng.integers(0, 4, size=(n, n)).astype(np.float64))
    if kind == "float32":
        return symmetric(rng.random((n, n)).astype(np.float32).astype(np.float64))
    if kind == "float64":  # Euclidean
        P = rng.random((n, 3))
        return np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    # KT-style: negative entries and duplicate rows
    P = rng.normal(size=(n, 4))
    P[n // 2: n // 2 + 3] = P[:3][: len(P[n // 2: n // 2 + 3])]
    return symmetric(np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1)) - 1.0)


def reference(D, method):
    return scipy_linkage(squareform(D, checks=False), method)


def not_a_tree(Z):
    """scipy's result after an all-NaN scan (ward on non-Euclidean data), where its nn_chain reuses a stale index:
    a cluster merged with itself, or a root that does not hold every point."""
    return bool((Z[:, 0] == Z[:, 1]).any() or Z[-1, 3] != len(Z) + 1)


@pytest.mark.parametrize("method", lo.METHODS)
@pytest.mark.parametrize("kind", ["ties", "float32", "float64", "kt"])
def test_oracle_equals_scipy_bit_for_bit(kind, method):
    refused = 0
    for seed in range(12):
        n = 2 + (7 * seed) % 45
        D = make(kind, n, seed)
        want = reference(D, method)
        try:
            got = lo.linkage(D, method)
        except ValueError:
            # ward on non-Euclidean data: a tip whose distances are all NaN; scipy then reuses a stale index
            # and returns a matrix that is not a tree (a cluster merged with itself)
            assert kind == "kt" and method == "ward"
            assert not_a_tree(want)
            refused += 1
            continue
        assert np.array_equal(got, want, equal_nan=True), (seed, n)
    assert refused < 12


@pytest.mark.parametrize("method", lo.METHODS)
@pytest.mark.parametrize("n", [2, 3])
def test_oracle_at_two_and_three_points(n, method):
    for D in (make("ties", n, 0), make("float64", n, 1), np.zeros((n, n))):
        assert np.array_equal(lo.linkage(D, method), reference(D, method))


def test_ward_nan_heights_are_reproduced():
    cases = 0
    for seed in range(40):
        D = make("kt", 30, seed)
        want = reference(D, "ward")
        if not np.isnan(want[:, 2]).any() or not_a_tree(want):
            continue
        assert np.array_equal(lo.linkage(D, "ward"), want, equal_nan=True)
        cases += 1
    assert cases > 0


@pytest.mark.parametrize("method", lo.METHODS)
def test_host_stage_sorts_and_labels_as_scipy(method):
    for seed in range(6):
        D = make("ties", 40 + seed, seed)
        raw = lo.prim_raw(D) if method == "single" else lo.nn_chain_raw(D, method)[0]
        Z = phyloselect.linkage_tree(raw[:, 0].astype(np.int64), raw[:, 1].astype(np.int64), raw[:, 2])
        assert np.array_equal(Z, reference(D, method))


def test_nn_chain_stays_within_its_scan_bound():
    for kind in ("ties", "float64"):
        D = make(kind, 200, 5)
        for method in ("complete", "average", "weighted", "ward"):
            assert lo.nn_chain_raw(D, method)[1] <= 3 * (200 - 1)


def parse_newick(text):
    """(parent, length, name) per node of a Newick string; the root is node 0 with parent -1."""
    parent, length, name = [], [], []

    def new(p):
        parent.append(p)
        length.append(0.0)
        name.append(None)
        return len(parent) - 1

    text = text.strip()
    assert text.endswith(";")
    text = text[:-1]
    stack, last, i = [], None, 0
    while i < len(text):
        c = text[i]
        if c == "(":
            node = new(stack[-1] if stack else -1)
            stack.append(node)
            i += 1
        elif c == ",":
            i += 1
        elif c == ")":
            last = stack.pop()
            i += 1
        elif c == ":":
            j = i + 1
            while j < len(text) and text[j] not in ",)":
                j += 1
            length[last] = float(text[i + 1:j])
            i = j
        else:
            if c == "'":
                buf, j = [], i + 1
                while True:
                    if text[j] == "'" and j + 1 < len(text) and text[j + 1] == "'":
                        buf.append("'")
                        j += 2
                    elif text[j] == "'":
                        j += 1
                        break
                    else:
                        buf.append(text[j])
                        j += 1
                label = "".join(buf)
            else:
                j = i
                while j < len(text) and text[j] not in ":,)":
                    j += 1
                label = text[i:j]
            last = new(stack[-1])
            name[last] = label
            i = j
    return np.array(parent), np.array(length), name


def leaf_path_lengths(parent, length, name, names):
    """Leaf-to-leaf path lengths, ordered as `names`, as a condensed vector."""
    depth = np.zeros(len(parent))
    for v in range(1, len(parent)):  # parents precede their children in a preorder
        depth[v] = depth[parent[v]] + length[v]
    leaf = {nm: v for v, nm in enumerate(name) if nm is not None}
    anc = []
    for nm in names:
        v, chain = leaf[nm], []
        while v != -1:
            chain.append(v)
            v = parent[v]
        anc.append(chain)
    n = len(names)
    out = []
    for a in range(n):
        sa = set(anc[a])
        for b in range(a + 1, n):
            lca = next(v for v in anc[b] if v in sa)
            out.append(depth[anc[a][0]] + depth[anc[b][0]] - 2 * depth[lca])
    return np.array(out)


@pytest.mark.parametrize("method", lo.METHODS)
def test_newick_round_trip_gives_the_cophenetic_distances(tmp_path, method):
    D = make("float64", 30, 9)
    Z = reference(D, method)
    names = ["c%d" % i for i in range(30)]
    path = tmp_path / "tree.nwk"
    phyloselect.write_newick(Z, names, str(path))
    parent, length, name = parse_newick(path.read_text())
    assert sorted(nm for nm in name if nm is not None) == sorted(names)
    assert (length[1:] >= 0).all()
    assert np.allclose(leaf_path_lengths(parent, length, name, names), cophenet(Z), rtol=1e-12, atol=1e-12)


def test_newick_of_a_deep_single_linkage_tree(tmp_path):
    n = 3000  # points on a line: every single-linkage merge adds one leaf, the tree is n deep
    x = np.cumsum(np.random.default_rng(0).random(n) + 0.5)
    D = np.abs(x[:, None] - x[None, :])
    Z = reference(D, "single")
    path = tmp_path / "deep.nwk"
    phyloselect.write_newick(Z, [str(i) for i in range(n)], str(path))
    parent, length, name = parse_newick(path.read_text())
    assert sum(nm is not None for nm in name) == n and len(parent) == 2 * n - 1


def test_newick_names_are_quoted_when_needed(tmp_path):
    names = ["plain_id", "with blank", "o'brien", "a(b)", "x:y", "p,q", "semi;", "[c]", "tab\tname", ""]
    assert [phyloselect.newick_name(s) for s in names] == [
        "plain_id", "'with blank'", "'o''brien'", "'a(b)'", "'x:y'", "'p,q'", "'semi;'", "'[c]'", "'tab\tname'", "''"]
    D = make("float64", len(names), 4)
    path = tmp_path / "q.nwk"
    phyloselect.write_newick(reference(D, "average"), names, str(path))
    _, _, parsed = parse_newick(path.read_text())
    assert sorted(nm for nm in parsed if nm is not None) == sorted(names)


def test_working_copy_size_test():
    n = 100_000
    need = phyloselect.linkage_bytes(n, "average")
    assert need >= 8 * n * n
    with pytest.raises(PhyloligoError, match=r"needs %d bytes" % need):
        phyloselect.check_linkage_fits(n, "average", 40 * 10**9)
    phyloselect.check_linkage_fits(n, "single", 40 * 10**9)  # single reads the matrix in place
    assert phyloselect.linkage_bytes(n, "single") < 10**8


@pytest.mark.parametrize("method", ["centroid", "median", "nj"])
def test_unsupported_methods_are_refused(method):
    with pytest.raises(ValueError, match="not supported" if method != "nj" else "must be one of"):
        phyloselect.linkage(np.zeros((4, 4)), method)
    with pytest.raises(ValueError):
        phyloselect.HClust(linkage=method)


def test_leaf_names_are_the_fasta_record_ids(tmp_path):
    path = tmp_path / "a.fa"
    path.write_bytes(b">ctg1 length=12 cov=3\nACGTACGTACGT\n>ctg(2)\r\nACGT\r\nAC\r\n>ctg3\tdesc\nAAAA\n")
    ids = phyloselect.fasta_record_ids(str(path))
    assert ids == ["ctg1", "ctg(2)", "ctg3"]
    assert [phyloselect.newick_name(s) for s in ids] == ["ctg1", "'ctg(2)'", "ctg3"]
