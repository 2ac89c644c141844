"""CPU ORACLE of phyloselect's HDBSCAN -- TEST INFRASTRUCTURE ONLY (never imported by phyloligo_b200/;
tests/ only).

numpy restatement of what hdbscan.HDBSCAN(min_cluster_size, min_samples, metric="precomputed") computes
with every other argument at its default (scikit-learn-contrib/hdbscan: ``mutual_reachability``,
``mst_linkage_core``, ``label``, ``condense_tree``, ``compute_stability``, ``get_clusters``,
``get_probabilities``), with one deliberate difference: MST edges compare by the triple
(mutual reachability, min(i, j), max(i, j)), which makes the MST unique and the result independent of a
Prim start vertex or an unstable sort.  Stages:

1. core distance of row i: the (min_samples + 1)-th smallest entry of the row, diagonal included
   (contrib: np.partition(D, min_samples, axis=0)[min_samples]); an entry of D in D's dtype;
2. mutual reachability mr(i, j) = max(core_i, core_j, D[i, j]);
3. MST of the complete mr graph under the tie rule: ``mst_kruskal`` (dense, N <= 3000) and
   ``mst_prim_streaming`` (one row of D at a time, for larger N);
4. single-linkage tree, condensed tree, stability, excess-of-mass selection, labels, probabilities.
"""
import numpy as np

CONDENSED_DTYPE = np.dtype([("parent", np.int64), ("child", np.int64), ("lambda_val", np.float64), ("child_size", np.int64)])


def clamp_min_samples(n, min_cluster_size, min_samples=None):
    ms = min_cluster_size if min_samples is None else min_samples
    return min(ms, n - 1)


def core_distances(D, min_samples):
    """contrib's np.partition(D, min_samples, axis=0)[min_samples] on a symmetric matrix, in D's dtype."""
    return np.partition(D, min_samples, axis=1)[:, min_samples]


def _orient(u, v, w):
    a, b = np.minimum(u, v), np.maximum(u, v)
    order = np.lexsort((b, a, w))
    return a[order].astype(np.int64), b[order].astype(np.int64), w[order]


def mst_kruskal(D, core):
    """Kruskal over the dense mr matrix under the tie rule.  Returns (u, v, w) in tie-rule order, u < v,
    w in D's dtype."""
    n = D.shape[0]
    iu, ju = np.triu_indices(n, 1)
    w = np.maximum(np.maximum(core[iu], core[ju]), D[iu, ju])
    order = np.lexsort((ju, iu, w))
    iu, ju, w = iu[order], ju[order], w[order]
    comp = np.arange(n)
    members = [[i] for i in range(n)]
    out = []
    chunk = 1 << 16
    for s in range(0, len(w), chunk):
        a, b = iu[s:s + chunk], ju[s:s + chunk]
        keep = np.nonzero(comp[a] != comp[b])[0]
        for q in keep:
            ca, cb = comp[a[q]], comp[b[q]]
            if ca == cb:
                continue
            if len(members[ca]) < len(members[cb]):
                ca, cb = cb, ca
            comp[members[cb]] = ca
            members[ca].extend(members[cb])
            members[cb] = []
            out.append(s + q)
        if len(out) == n - 1:
            break
    out = np.asarray(out, dtype=np.int64)
    return _orient(iu[out], ju[out], w[out])


def mst_prim_streaming(D, core):
    """Prim under the tie rule reading one row of D per step (D may be a memmap or any row-indexable
    array); O(N) memory besides D.  Same result as ``mst_kruskal``: the MST under a strict total order
    of the edges is unique."""
    n = D.shape[0]
    in_tree = np.zeros(n, dtype=bool)
    best_w = np.full(n, np.inf)
    best_u = np.full(n, -1, dtype=np.int64)
    idx = np.arange(n)
    cur = 0
    in_tree[0] = True
    us, vs, ws = [], [], []
    for _ in range(n - 1):
        row = np.asarray(D[cur])
        cand = np.maximum(np.maximum(core[cur], core), row).astype(np.float64)
        # tie rule: (w, min(cur, v), max(cur, v)) against (best_w, min(best_u, v), max(best_u, v))
        cmin, cmax = np.minimum(cur, idx), np.maximum(cur, idx)
        bmin, bmax = np.minimum(best_u, idx), np.maximum(best_u, idx)
        better = (cand < best_w) | ((cand == best_w) & ((cmin < bmin) | ((cmin == bmin) & (cmax < bmax))))
        better &= ~in_tree
        best_w = np.where(better, cand, best_w)
        best_u = np.where(better, cur, best_u)
        out = np.nonzero(~in_tree)[0]
        bw = best_w[out]
        m = bw.min()
        tied = out[bw == m]
        tmin, tmax = np.minimum(best_u[tied], tied), np.maximum(best_u[tied], tied)
        pick = tied[np.lexsort((tmax, tmin))[0]]
        us.append(best_u[pick])
        vs.append(pick)
        ws.append(max(core[best_u[pick]], core[pick], D[best_u[pick], pick]))
        in_tree[pick] = True
        cur = pick
    return _orient(np.asarray(us, dtype=np.int64), np.asarray(vs, dtype=np.int64), np.asarray(ws, dtype=D.dtype))


def single_linkage(u, v, w, n):
    """contrib's label(): edges in tie-rule order; rows (left, right, distance, size)."""
    parent = np.arange(2 * n - 1)
    size = np.ones(2 * n - 1, dtype=np.int64)

    def find(x):
        r = x
        while parent[r] != r:
            r = parent[r]
        while parent[x] != r:
            parent[x], x = r, parent[x]
        return r

    left = np.empty(n - 1, dtype=np.int64)
    right = np.empty(n - 1, dtype=np.int64)
    sizes = np.empty(n - 1, dtype=np.int64)
    nxt = n
    for k in range(n - 1):
        a, b = find(int(u[k])), find(int(v[k]))
        left[k], right[k] = a, b
        sizes[k] = size[a] + size[b]
        parent[a] = parent[b] = nxt
        size[nxt] = sizes[k]
        nxt += 1
    return left, right, np.asarray(w, dtype=np.float64), sizes


def _bfs(left, right, n, root):
    out, queue = [], [root]
    while queue:
        out.extend(queue)
        nxt = []
        for x in queue:
            if x >= n:
                nxt.extend((left[x - n], right[x - n]))
        queue = nxt
    return out


def condense_tree(left, right, dist, sizes, n, min_cluster_size):
    """contrib's condense_tree()."""
    root = 2 * n - 2
    next_label = n + 1
    relabel = np.empty(root + 1, dtype=np.int64)
    relabel[root] = n
    ignore = np.zeros(root + 1, dtype=bool)
    rows = []

    def count(x):
        return sizes[x - n] if x >= n else 1

    for node in _bfs(left, right, n, root):
        if ignore[node] or node < n:
            continue
        l, r, d = left[node - n], right[node - n], dist[node - n]
        lam = 1.0 / d if d > 0.0 else np.inf
        lc, rc = count(l), count(r)
        if lc >= min_cluster_size and rc >= min_cluster_size:
            relabel[l] = next_label
            next_label += 1
            rows.append((relabel[node], relabel[l], lam, lc))
            relabel[r] = next_label
            next_label += 1
            rows.append((relabel[node], relabel[r], lam, rc))
        else:
            if lc < min_cluster_size and rc >= min_cluster_size:
                relabel[r] = relabel[node]
                drop = [l]
            elif rc < min_cluster_size and lc >= min_cluster_size:
                relabel[l] = relabel[node]
                drop = [r]
            else:
                drop = [l, r]
            for sub in drop:
                for s in _bfs(left, right, n, sub):
                    if s < n:
                        rows.append((relabel[node], s, lam, 1))
                    ignore[s] = True
    return np.array(rows, dtype=CONDENSED_DTYPE)


def compute_stability(ct):
    """contrib's compute_stability(): {cluster id: stability}, accumulated in condensed-tree order."""
    smallest = int(ct["parent"].min())
    largest_child = max(int(ct["child"].max()), smallest)
    births = np.full(largest_child + 1, np.nan)
    births[ct["child"]] = ct["lambda_val"]
    births[smallest] = 0.0
    num = int(ct["parent"].max()) - smallest + 1
    result = np.zeros(num)
    for p, lam, sz in zip(ct["parent"].tolist(), ct["lambda_val"].tolist(), ct["child_size"].tolist()):
        result[p - smallest] += (lam - births[p]) * sz
    return {smallest + i: result[i] for i in range(num)}


def get_clusters(ct, stability, n):
    """contrib's get_clusters() with cluster_selection_method="eom", allow_single_cluster=False:
    (labels int64, probabilities float64)."""
    node_list = sorted(stability.keys(), reverse=True)[:-1]
    cluster_rows = ct[ct["child_size"] > 1]
    children = {}
    for p, c in zip(cluster_rows["parent"].tolist(), cluster_rows["child"].tolist()):
        children.setdefault(p, []).append(c)
    is_cluster = {c: True for c in node_list}
    for node in node_list:
        kids = children.get(node, [])
        subtree = np.sum([stability[c] for c in kids])
        if subtree > stability[node]:
            is_cluster[node] = False
            stability[node] = subtree
        else:
            queue = list(kids)
            while queue:
                x = queue.pop()
                is_cluster[x] = False
                queue.extend(children.get(x, []))
    clusters = sorted(c for c in is_cluster if is_cluster[c])
    label_of = {c: i for i, c in enumerate(clusters)}
    root = int(ct["parent"].min())
    # a point's label is its nearest selected ancestor in the condensed tree (contrib's do_labelling)
    top = {root: -1}
    for p, c in zip(cluster_rows["parent"].tolist(), cluster_rows["child"].tolist()):
        top[c] = label_of[c] if c in label_of else top[p]
    labels = np.full(n, -1, dtype=np.int64)
    points = ct[ct["child"] < n]
    labels[points["child"]] = [top[p] for p in points["parent"].tolist()]
    # contrib's get_probabilities(): lambda over the cluster's largest lambda
    deaths = {}
    for p, lam in zip(ct["parent"].tolist(), ct["lambda_val"].tolist()):
        deaths[p] = max(deaths.get(p, lam), lam)
    probs = np.zeros(n)
    for c, lam in zip(points["child"].tolist(), points["lambda_val"].tolist()):
        if labels[c] == -1:
            continue
        ml = deaths[clusters[labels[c]]]
        probs[c] = 1.0 if (ml == 0.0 or not np.isfinite(lam)) else min(lam, ml) / ml
    return labels, probs


def tree_to_labels(u, v, w, n, min_cluster_size):
    """Stage 4 from an MST in tie-rule order: (labels, probabilities, condensed tree, single-linkage rows)."""
    sl = single_linkage(u, v, w, n)
    ct = condense_tree(*sl, n, min_cluster_size)
    labels, probs = get_clusters(ct, compute_stability(ct), n)
    return labels, probs, ct, sl


def hdbscan(D, min_cluster_size=5, min_samples=None):
    """Every stage on a dense symmetric matrix: dict with core, mst (u, v, w), labels, probabilities,
    condensed tree."""
    n = D.shape[0]
    ms = clamp_min_samples(n, min_cluster_size, min_samples)
    core = core_distances(D, ms)
    u, v, w = mst_kruskal(D, core)
    labels, probs, ct, _ = tree_to_labels(u, v, w, n, min_cluster_size)
    return {"core": core, "mst": (u, v, w), "labels": labels, "probabilities": probs, "condensed_tree": ct}
