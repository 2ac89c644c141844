"""numpy restatement of scipy.cluster.hierarchy.linkage(squareform(D, checks=False), method) for the methods
phyloselect.linkage supports (scipy 1.18.1, cluster/_hierarchy.pyx; its .pyx source is not installed with scipy).

- complete / average / weighted / ward: ``nn_chain``.  The tip x scans the active clusters i != x in ascending
  order and takes i only if d(x, i) < cur, cur starting at d(x, prev) (prev: the entry below the tip) or +inf on a
  one-entry chain.  y == prev merges x and y (swapped so that x < y; the new cluster lives in slot y), otherwise
  y is pushed.  An empty chain takes the lowest-index active cluster.
- single: ``mst_single_linkage``, Prim from vertex 0.
- both: a stable argsort of the heights, then ``label`` (union-find; new clusters n, n + 1, ...).

All arithmetic is float64 on the float64 copy of the entries, comparisons are IEEE < and > (false on NaN), and
the Lance-Williams updates are written operation by operation as scipy's C evaluates them.
"""
import numpy as np

METHODS = ("single", "complete", "average", "weighted", "ward")


def update(method, dxi, dyi, dxy, nx, ny, ni):
    """scipy's _hierarchy_distance_update.pxi for one cluster i (sizes are Python ints)."""
    if method == "complete":
        return dyi if dyi > dxi else dxi
    if method == "average":
        return (nx * dxi + ny * dyi) / (nx + ny)
    if method == "weighted":
        return 0.5 * (dxi + dyi)
    t = 1.0 / (nx + ny + ni)
    with np.errstate(invalid="ignore"):
        return np.sqrt((ni + nx) * t * dxi * dxi + (ni + ny) * t * dyi * dyi - ni * t * dxy * dxy)


def _first_min_below(row, cand, cur):
    """The sequential scan `if row[i] < cur: cur, y = row[i], i` over the indices `cand` (ascending): (y, cur),
    y None when nothing is taken."""
    vals = row[cand]
    take = vals < cur
    if not take.any():
        return None, cur
    v = vals[take]
    m = v.min()
    return int(cand[take][np.flatnonzero(v == m)[0]]), m


def nn_chain_raw(D, method):
    """The n - 1 raw merges (x, y, height) of scipy's nn_chain in merge order, and the number of scans."""
    W = np.array(D, dtype=np.float64)
    n = len(W)
    size = np.ones(n, np.int64)
    raw = []
    chain = []
    y = 0  # scipy keeps y across scans
    scans = 0
    for _ in range(n - 1):
        if not chain:
            chain = [int(np.flatnonzero(size > 0)[0])]
        while True:
            x = chain[-1]
            cand = np.flatnonzero(size > 0)
            cand = cand[cand != x]
            if len(chain) > 1:
                prev = chain[-2]
                y, cur = prev, W[x, prev]
            else:
                cur = np.inf
            j, cur = _first_min_below(W[x], cand, cur)
            scans += 1
            if j is not None:
                y = j
            elif len(chain) == 1 and (y == x or size[y] == 0):
                raise ValueError("every distance from the chain's tip is NaN")
            if len(chain) > 1 and y == chain[-2]:
                break
            chain.append(y)
        chain.pop()
        chain.pop()
        if x > y:
            x, y = y, x
        nx, ny = int(size[x]), int(size[y])
        raw.append((x, y, cur))
        size[x] = 0
        size[y] = nx + ny
        for i in np.flatnonzero(size > 0):
            if i == y:
                continue
            W[i, y] = W[y, i] = update(method, W[i, x], W[i, y], cur, nx, ny, int(size[i]))
    return np.array(raw, dtype=np.float64).reshape(-1, 3), scans


def prim_raw(D):
    """The n - 1 raw steps (x, y, height) of scipy's mst_single_linkage."""
    D = np.asarray(D, dtype=np.float64)
    n = len(D)
    best = np.full(n, np.inf)
    merged = np.zeros(n, bool)
    raw = []
    x = 0
    for _ in range(n - 1):
        merged[x] = True
        cand = np.flatnonzero(~merged)
        row = D[x, cand]
        upd = best[cand] > row
        best[cand[upd]] = row[upd]
        y, cur = _first_min_below(best, cand, np.inf)
        raw.append((x, y, cur))
        x = y
    return np.array(raw, dtype=np.float64).reshape(-1, 3)


def finish(raw, n):
    """Stable sort by height (NaN last) and scipy's label: the (n - 1, 4) linkage matrix."""
    raw = raw[np.argsort(raw[:, 2], kind="mergesort")]
    parent = np.arange(2 * n - 1)
    size = np.ones(2 * n - 1, np.int64)

    def find(a):
        r = a
        while parent[r] != r:
            r = parent[r]
        while parent[a] != r:
            parent[a], a = r, parent[a]
        return r

    Z = np.empty((n - 1, 4))
    for k, (x, y, h) in enumerate(raw):
        a, b = sorted((find(int(x)), find(int(y))))
        parent[a] = parent[b] = n + k
        size[n + k] = size[a] + size[b]
        Z[k] = a, b, h, size[n + k]
    return Z


def linkage(D, method):
    """scipy.cluster.hierarchy.linkage(squareform(D, checks=False), method), bit for bit."""
    n = len(D)
    raw = prim_raw(D) if method == "single" else nn_chain_raw(D, method)[0]
    return finish(raw, n)
