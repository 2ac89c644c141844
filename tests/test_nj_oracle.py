"""The neighbour-joining restatement (oracle/nj_oracle.py) and the Newick writer of phyloselect.nj on the CPU:
textbook lengths, recovery of additive trees, the tie rule and the Newick round trip."""
import re

import numpy as np
import pytest

from oracle import nj_oracle
from phyloligo_b200 import phyloselect

TEXTBOOK = np.array([[0, 5, 9, 9, 8], [5, 0, 10, 10, 9], [9, 10, 0, 8, 7], [9, 10, 8, 0, 3], [8, 9, 7, 3, 0]], dtype=np.float64)


def random_tree(n, seed):
    """A seeded random binary tree by random merges of clades, branch lengths in [0.05, 1].  Returns its patristic
    distance matrix and its splits {frozenset of the side without leaf 0: length} of the unrooted tree (the two
    branches at the root are one edge)."""
    rng = np.random.default_rng(seed)
    D = np.zeros((n, n))
    depth = np.zeros(n)
    clades = [[i] for i in range(n)]
    splits = {}
    while len(clades) > 2:
        i, j = sorted(rng.choice(len(clades), 2, replace=False))
        A, B = clades[i], clades[j]
        la, lb = rng.uniform(0.05, 1.0, 2)
        depth[A] += la
        depth[B] += lb
        D[np.ix_(A, B)] = depth[A][:, None] + depth[B][None, :]
        D[np.ix_(B, A)] = D[np.ix_(A, B)].T
        for side, ln in ((A, la), (B, lb)):
            splits[canonical(side, n)] = ln
        clades = [c for k, c in enumerate(clades) if k not in (i, j)] + [A + B]
    A, B = clades
    ln = rng.uniform(0.05, 1.0)
    D[np.ix_(A, B)] = depth[A][:, None] + depth[B][None, :] + ln
    D[np.ix_(B, A)] = D[np.ix_(A, B)].T
    key = canonical(A, n)
    splits[key] = splits.get(key, 0.0) + ln  # A's own branch (if A was merged) and the root edge are one edge
    return D, splits


def canonical(side, n):
    s = frozenset(int(x) for x in side)
    return s if 0 not in s else frozenset(range(n)) - s


def tree_splits(edge, length, n):
    """{canonical split: length} of every edge of an nj tree (rooted at n for the walk)."""
    children = {}
    for (p, c), ln in zip(edge.tolist(), length.tolist()):
        children.setdefault(p, []).append((c, ln))
    leaves = {}
    order, stack = [], [n]
    while stack:
        v = stack.pop()
        order.append(v)
        stack += [c for c, _ in children.get(v, [])]
    for v in reversed(order):
        leaves[v] = {v} if v < n else set().union(*(leaves[c] for c, _ in children[v]))
    out = {}
    for (p, c), ln in zip(edge.tolist(), length.tolist()):
        key = canonical(leaves[c], n)
        out[key] = out.get(key, 0.0) + ln
    return out


def check_shape(edge, length, n):
    assert edge.shape == (2 * n - 3, 2) and edge.dtype == np.int64 and length.shape == (2 * n - 3,)
    # every node but the root is a child exactly once; the root has three children, a joined node two
    assert sorted(edge[:, 1].tolist()) == [i for i in range(2 * n - 2) if i != n]
    parents, counts = np.unique(edge[:, 0], return_counts=True)
    assert dict(zip(parents.tolist(), counts.tolist())) == {p: (3 if p == n else 2) for p in range(n, 2 * n - 2)}


@pytest.mark.parametrize("method", ["nj", "bionj"])
def test_textbook_five_taxa(method):
    edge, length = nj_oracle.nj(TEXTBOOK, method)
    check_shape(edge, length, 5)
    assert edge.tolist() == [[7, 0], [7, 1], [6, 7], [6, 2], [5, 6], [5, 3], [5, 4]]
    assert length.tolist() == [2.0, 3.0, 3.0, 4.0, 2.0, 2.0, 1.0]


@pytest.mark.parametrize("method", ["nj", "bionj"])
@pytest.mark.parametrize("n,seed", [(4, 1), (7, 2), (12, 3), (40, 4), (150, 5)])
def test_additive_tree_recovered(n, seed, method):
    D, want = random_tree(n, seed)
    edge, length = nj_oracle.nj(D, method)
    check_shape(edge, length, n)
    got = tree_splits(edge, length, n)
    assert set(got) == set(want)  # Robinson-Foulds distance 0
    assert max(abs(got[k] - want[k]) for k in want) <= 1e-9


def test_bionj_equals_nj_on_additive_data():
    D, _ = random_tree(60, 11)
    e1, l1 = nj_oracle.nj(D, "nj")
    e2, l2 = nj_oracle.nj(D, "bionj")
    assert tree_splits(e1, l1, 60).keys() == tree_splits(e2, l2, 60).keys()
    a, b = tree_splits(e1, l1, 60), tree_splits(e2, l2, 60)
    assert max(abs(a[k] - b[k]) for k in a) <= 1e-9


@pytest.mark.parametrize("method", ["nj", "bionj"])
def test_three_rows(method):
    D = np.array([[0.0, 3.0, 4.0], [3.0, 0.0, 5.0], [4.0, 5.0, 0.0]])
    edge, length = nj_oracle.nj(D, method)
    assert edge.tolist() == [[3, 0], [3, 1], [3, 2]]
    assert length.tolist() == [1.0, 2.0, 3.0]


def test_ties_resolve_by_list_position():
    # split {0, 3} | {1, 2} with integer lengths: Q(0, 3) == Q(1, 2) exactly, the smallest; (0, 3) comes first
    D = np.array([[0, 8, 6, 3], [8, 0, 4, 9], [6, 4, 0, 7], [3, 9, 7, 0]], dtype=np.float64)
    edge, _ = nj_oracle.nj(D, "nj")
    assert edge[:2].tolist() == [[5, 0], [5, 3]]
    # the same matrix with rows 0 and 1 swapped: now (0, 2) and (1, 3) tie, (0, 2) comes first
    p = [1, 0, 2, 3]
    edge, _ = nj_oracle.nj(D[np.ix_(p, p)], "nj")
    assert edge[:2].tolist() == [[5, 0], [5, 2]]
    # all distances equal: every Q ties, the first pair (0, 1) is taken, then the new node (list position 0) with 2
    E = np.ones((6, 6)) - np.eye(6)
    edge, _ = nj_oracle.nj(E, "nj")
    assert edge[:4].tolist() == [[9, 0], [9, 1], [8, 9], [8, 2]]


def test_row_sums_are_sequential_in_rotated_order():
    rng = np.random.default_rng(3)
    M = rng.normal(size=(9, 9)) * 10.0 ** rng.integers(-8, 8, size=(9, 9))
    S = nj_oracle.row_sums(M)
    for a in range(9):
        s = 0.0
        for b in list(range(a + 1, 9)) + list(range(a)):
            s += M[a, b]
        assert S[a] == s


def parse_newick(text):
    """(splits {canonical split: length} keyed by leaf name sets, leaf names in order) of an unrooted Newick tree
    with single-quoted names allowed."""
    tokens = re.findall(r"'(?:[^']|'')*'|[(),:;]|[^(),:;']+", text.strip())
    stack, groups, names = [[]], [], []
    i = 0
    while i < len(tokens):
        tok = tokens[i]
        if tok == "(":
            stack.append([])
        elif tok == ")":
            members = stack.pop()
            leafset = set().union(*(m for m, _ in members))
            groups += members
            stack[-1].append([leafset, None])
        elif tok in (",", ";"):
            pass
        elif tok == ":":
            stack[-1][-1][1] = float(tokens[i + 1])
            i += 1
        else:
            name = tok[1:-1].replace("''", "'") if tok.startswith("'") else tok
            names.append(name)
            stack[-1].append([{name}, None])
        i += 1
    return groups, names


def test_write_nj_newick_round_trip(tmp_path):
    n = 30
    D, _ = random_tree(n, 8)
    edge, length = nj_oracle.nj(D, "nj")
    names = ["c%d" % i for i in range(n)]
    names[3] = "odd name"
    names[5] = "it's"
    path = tmp_path / "t.nwk"
    phyloselect.write_nj_newick(edge, length, names, str(path))
    text = path.read_text()
    assert text.endswith(";\n") and "'odd name'" in text and "'it''s'" in text
    groups, order = parse_newick(text)
    assert sorted(order) == sorted(names)
    index = {name: i for i, name in enumerate(names)}
    got = {}
    for leafset, ln in groups:
        key = canonical([index[x] for x in leafset], n)
        got[key] = got.get(key, 0.0) + ln
    want = tree_splits(edge, length, n)
    assert got.keys() == want.keys()
    assert all(got[k] == want[k] for k in want)  # repr(float) round-trips exactly, and each edge is written once
    # the root is trifurcating: its three children are the root edges, in order
    top = text[1:text.rindex(")")]
    depth, parts, cur = 0, [], ""
    for ch in top:
        if ch == "," and depth == 0:
            parts.append(cur)
            cur = ""
            continue
        depth += ch == "("
        depth -= ch == ")"
        cur += ch
    parts.append(cur)
    assert len(parts) == 3
    assert [float(p.rsplit(":", 1)[1]) for p in parts] == length[-3:].tolist()


def test_write_nj_newick_caterpillar_is_iterative(tmp_path):
    # a caterpillar tree deeper than Python's recursion limit
    n = 3000
    edge = []
    length = []
    prev = 0
    for t in range(n - 3):
        u = 2 * n - 3 - t
        edge += [(u, prev), (u, t + 1)]
        length += [1.0, 0.5]
        prev = u
    edge += [(n, prev), (n, n - 2), (n, n - 1)]
    length += [1.0, 0.5, 0.25]
    path = tmp_path / "cat.nwk"
    phyloselect.write_nj_newick(np.array(edge), np.array(length), [str(i) for i in range(n)], str(path))
    text = path.read_text()
    assert text.count("(") == n - 2 and text.count(",") == n - 1  # n - 3 joined nodes, one comma each; the root two


def test_write_nj_newick_refuses_bad_shapes(tmp_path):
    edge, length = nj_oracle.nj(TEXTBOOK, "nj")
    with pytest.raises(ValueError, match="names"):
        phyloselect.write_nj_newick(edge, length, ["a", "b"], str(tmp_path / "x.nwk"))


def test_oracle_refusals():
    with pytest.raises(ValueError, match="at least 3"):
        nj_oracle.nj(np.zeros((2, 2)))
    with pytest.raises(ValueError, match="method"):
        nj_oracle.nj(TEXTBOOK, "upgma")
    with pytest.raises(ValueError, match="1e50"):
        nj_oracle.nj(np.full((4, 4), -1e60) + np.diag(np.full(4, 1e60)))  # every Q is 4e60, above ape's bound
