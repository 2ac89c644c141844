"""numpy restatement of the neighbour-joining trees phyloselect.R builds with ape's ``nj`` and ``bionj``, with the
order of every float64 operation fixed.  ``phyloselect.nj`` on the device equals it bit for bit.

NJ (ape's nj.c as far as it can be restated without its source).  An ordered active list L starts as 0 .. n-1.
While m = |L| > 3:

1. S_a, for every a in L, is a sequential float64 sum from 0: the distances to the members after a in list order,
   then those before a in list order (ape's sum_dist_to_i over its condensed array).  numpy's ``sum`` is pairwise,
   so the sums here are ``cumsum`` over the rotated rows, which adds in order.
2. Q(a, b) = ((m - 2) d(a, b) - S_a) - S_b for a before b.  The pair taken has the strictly smallest Q below the
   starting bound 1e50; on ties the first pair in lexicographic order of list positions.
3. A = d(a, b), B = (S_a - S_b) / (m - 2); the branch lengths are (A + B) / 2 for a and (A - B) / 2 for b, and the
   new node u has d(u, k) = ((d(a, k) + d(b, k)) - A) / 2.
4. L <- [u] + (L without a, b).

With three members x, y, z left the root edges are ((d_xy + d_xz) - d_yz) / 2, ((d_xy + d_yz) - d_xz) / 2 and
((d_yz + d_xz) - d_xy) / 2.

BIONJ (Gascuel 1997) selects, sums and measures branches as NJ does on D, and keeps a variance matrix V, initially
D.  lambda = 1/2 + sum_k (V_bk - V_ak) / ((2 (m - 2)) V_ab), the sum sequential over the other members in list
order, lambda = 1/2 when V_ab = 0, then clipped to [0, 1];
d(u, k) = lambda (d_ak - l_a) + (1 - lambda)(d_bk - l_b);  V(u, k) = (lambda V_ak + (1 - lambda) V_bk) - (lambda (1 - lambda)) V_ab.

Agreement with ape is not pinned: neither R nor ape's C source has been available to compare against, and ape's
bionj is Gascuel's own program, whose pair order and tie tolerance are not restated here.

Output numbering is ape's, from 0: leaves 0 .. n-1, the root n, the node of join t (t = 0, 1, ...) 2n - 3 - t.
``edge`` rows are (parent, child) in join order, the first-listed member first, then the three root edges in list
order.
"""
import numpy as np

BOUND = 1e50


def _seq_sum(R):
    """Sequential float64 sums of the rows of R, each starting from +0.0 (numpy's cumsum adds in order)."""
    return np.cumsum(np.concatenate([np.zeros((R.shape[0], 1)), R], axis=1), axis=1)[:, -1]


def row_sums(M):
    """S_a for every list position a of the list-ordered matrix M: after a, then before a, in list order.  Row a
    of the strided view over [M | M] (with the diagonal of the first copy set to +0.0) starts at that 0 and runs
    through M[a, a+1:], then M[a, :a]."""
    m = len(M)
    B = np.empty((m, 2 * m))
    B[:, :m] = M
    B[:, m:] = M
    B[np.arange(m), np.arange(m)] = 0.0
    R = np.lib.stride_tricks.as_strided(B, shape=(m, m), strides=((2 * m + 1) * 8, 8), writeable=False)
    return np.cumsum(R, axis=1)[:, -1]


def select_pair(M, S, upper):
    """(a, b) list positions of the pair with the smallest Q below 1e50, the first in lexicographic order on ties.
    `upper` is a boolean matrix of at least m rows, True above the diagonal."""
    m = len(M)
    with np.errstate(invalid="ignore", over="ignore"):
        Q = ((m - 2.0) * M - S[:, None]) - S[None, :]
    Q = np.where(upper[:m, :m] & (Q < BOUND), Q, np.inf)  # NaN and the bound are never taken
    k = int(np.argmin(Q))  # the first minimum in row-major order: lexicographic in list positions
    if not Q.flat[k] < BOUND:
        raise ValueError("no pair has Q below 1e50 with %d members left" % m)
    return k // m, k % m


def nj(D, method="nj"):
    """(edge int64 (2n - 3, 2), length float64 (2n - 3,)) of NJ or BIONJ on the square matrix D (float32 values
    are widened exactly)."""
    if method not in ("nj", "bionj"):
        raise ValueError("method must be 'nj' or 'bionj', got {!r}".format(method))
    M = np.array(D, dtype=np.float64)
    n = len(M)
    if M.ndim != 2 or M.shape != (n, n) or n < 3:
        raise ValueError("a square matrix of at least 3 rows is expected, got shape {}".format(M.shape))
    V = M.copy() if method == "bionj" else None
    L = list(range(n))
    edge = np.empty((2 * n - 3, 2), np.int64)
    length = np.empty(2 * n - 3)
    upper = np.arange(n)[:, None] < np.arange(n)[None, :]
    t = 0
    with np.errstate(invalid="ignore", over="ignore"):
        while len(L) > 3:
            m = len(L)
            S = row_sums(M)
            a, b = select_pair(M, S, upper)
            A = M[a, b]
            B = (S[a] - S[b]) / (m - 2.0)
            la = (A + B) / 2.0
            lb = (A - B) / 2.0
            u = 2 * n - 3 - t
            edge[2 * t] = u, L[a]
            edge[2 * t + 1] = u, L[b]
            length[2 * t], length[2 * t + 1] = la, lb
            rest = np.r_[0:a, a + 1:b, b + 1:m]
            if V is None:
                du = ((M[a, rest] + M[b, rest]) - A) / 2.0
            else:
                Vab = V[a, b]
                if Vab == 0.0:
                    lam = 0.5
                else:
                    lam = 0.5 + _seq_sum((V[b, rest] - V[a, rest])[None, :])[0] / ((2.0 * (m - 2)) * Vab)
                    lam = 0.0 if lam < 0.0 else (1.0 if lam > 1.0 else lam)
                du = lam * (M[a, rest] - la) + (1.0 - lam) * (M[b, rest] - lb)
                vu = (lam * V[a, rest] + (1.0 - lam) * V[b, rest]) - (lam * (1.0 - lam)) * Vab
                V = _grow(V, a, b, vu)
            M = _grow(M, a, b, du)
            L = [u] + [L[k] for k in rest]
            t += 1
        x, y, z = L
        dxy, dxz, dyz = M[0, 1], M[0, 2], M[1, 2]
        edge[2 * t:] = [(n, x), (n, y), (n, z)]
        length[2 * t:] = ((dxy + dxz) - dyz) / 2.0, ((dxy + dyz) - dxz) / 2.0, ((dyz + dxz) - dxy) / 2.0
    return edge, length


def _grow(M, a, b, du):
    """The list-ordered matrix of [u] + (the members but a < b), du the distances of u to the others."""
    m = len(M)
    keep = [(0, a), (a + 1, b), (b + 1, m)]
    out = np.empty((m - 1, m - 1))
    out[0, 1:] = out[1:, 0] = du
    out[0, 0] = 0.0
    r = 1
    for r0, r1 in keep:
        c = 1
        for c0, c1 in keep:
            out[r:r + r1 - r0, c:c + c1 - c0] = M[r0:r1, c0:c1]
            c += c1 - c0
        r += r1 - r0
    return out
