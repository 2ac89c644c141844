"""float64 numpy restatement of scikit-learn 1.9's TSNE(metric="precomputed", method="barnes_hut", angle=0.0,
init="random"), the reference's -t projection (bin/phyloselect.py:381-398).  With angle 0 scikit-learn's
Barnes-Hut gradient is the exact gradient of the sparse-P objective, which is what this file computes:

  neighbours    k = min(n - 1, int(3 perplexity + 1)) per row, the row's own column excluded, squared in the
                matrix's dtype, then float32 (distances_nn.data **= 2; _joint_probabilities_nn)
  conditional   _binary_search_perplexity: float64, tolerance 1e-5 on the entropy, at most 100 steps
  joint P       (C + C^T) / sum, pairs whose sum is 0 dropped (scipy's sparse addition)
  gradient      4 (sum_j p_ij q_ij (y_i - y_j) - sum_j q_ij^2 (y_i - y_j) / Z), p_ij read as float32, exact
                over all pairs in row chunks (memory bounded)
  optimiser     _gradient_descent as _tsne drives it: 250 iterations with P x early_exaggeration and momentum 0.5,
                then momentum 0.8; gains +0.2 / x0.8 clipped at 0.01; a convergence check every 50 iterations
"""
import numpy as np
from scipy.sparse import csr_matrix

FLOAT32_TINY = float(np.finfo(np.float32).tiny)


def neighbours(D, perplexity):
    """(idx [n, k], squared float32 distances [n, k]) by a stable sort of every row without its own column."""
    D = np.asarray(D)
    n = D.shape[0]
    k = min(n - 1, int(3.0 * perplexity + 1))
    key = D.astype(np.float64, copy=True)
    np.fill_diagonal(key, np.inf)
    idx = np.argsort(key, axis=1, kind="stable")[:, :k]
    d = np.take_along_axis(D, idx, axis=1)
    return idx, (d * d).astype(np.float32)


def conditional(sq, perplexity, steps=100, tol=1e-5):
    """_binary_search_perplexity, all rows at once (each row stops at its own convergence)."""
    d = sq.astype(np.float64)
    n = d.shape[0]
    want = np.log(perplexity)
    beta = np.ones(n)
    lo = np.full(n, -np.inf)
    hi = np.full(n, np.inf)
    P = np.zeros_like(d)
    active = np.ones(n, dtype=bool)
    for _ in range(steps):
        a = np.nonzero(active)[0]
        if a.size == 0:
            break
        p = np.exp(-d[a] * beta[a, None])
        s = p.sum(axis=1)
        s[s == 0.0] = 1e-8
        p /= s[:, None]
        P[a] = p
        diff = np.log(s) + beta[a] * (d[a] * p).sum(axis=1) - want
        done = np.abs(diff) <= tol
        up = (diff > 0) & ~done
        down = (diff <= 0) & ~done
        b = beta[a].copy()
        lo_a, hi_a = lo[a].copy(), hi[a].copy()
        lo_a[up] = b[up]
        b[up] = np.where(hi_a[up] == np.inf, b[up] * 2.0, (b[up] + hi_a[up]) / 2.0)
        hi_a[down] = b[down]
        b[down] = np.where(lo_a[down] == -np.inf, b[down] / 2.0, (b[down] + lo_a[down]) / 2.0)
        beta[a], lo[a], hi[a] = b, lo_a, hi_a
        active[a[done]] = False
    return P


def joint_probabilities(D, perplexity):
    """The symmetric CSR P (float64, columns ascending)."""
    n = np.asarray(D).shape[0]
    idx, sq = neighbours(D, perplexity)
    C = conditional(sq, perplexity)
    k = idx.shape[1]
    Cm = csr_matrix((C.ravel(), idx.ravel(), np.arange(0, n * k + 1, k)), shape=(n, n))
    P = (Cm + Cm.T).tocsr()
    P.sort_indices()
    P.eliminate_zeros()
    P.data /= max(P.data.sum(), np.finfo(np.float64).eps)
    return P


def gradient(P, Y, exaggeration=1.0, chunk=512):
    """(grad float64 [n, 2], KL) at Y for P * exaggeration read as float32; the repulsion summed exactly over all
    pairs, `chunk` rows at a time."""
    Y = np.asarray(Y, dtype=np.float64)
    n = Y.shape[0]
    p32 = (P.data * exaggeration).astype(np.float32).astype(np.float64)
    rep = np.zeros((n, 2))
    Z = 0.0
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        diff = Y[r0:r1, None, :] - Y[None, :, :]
        q = 1.0 / (1.0 + (diff ** 2).sum(-1))
        q[np.arange(r1 - r0), np.arange(r0, r1)] = 0.0
        Z += q.sum()
        rep[r0:r1] = ((q * q)[:, :, None] * diff).sum(1)
    rows = np.repeat(np.arange(n), np.diff(P.indptr))
    b = Y[rows] - Y[P.indices]
    qa = 1.0 / (1.0 + (b ** 2).sum(-1))
    att = np.zeros((n, 2))
    np.add.at(att, rows, (p32 * qa)[:, None] * b)
    kl = float((p32 * np.log(np.maximum(p32, FLOAT32_TINY) / np.maximum(qa / Z, FLOAT32_TINY))).sum())
    return 4.0 * (att - rep / Z), kl


def random_init(n, random_state):
    """TSNE(init="random")'s draw."""
    rs = random_state if isinstance(random_state, np.random.RandomState) else np.random.RandomState(random_state)
    return 1e-4 * rs.standard_normal(size=(n, 2)).astype(np.float32)


def _descend(P, p, it, max_iter, momentum, lr, exaggeration, n_iter_without_progress, min_grad_norm, n_iter_check=50):
    update = np.zeros_like(p)
    gains = np.ones_like(p)
    error = best_error = np.finfo(float).max
    best_iter = i = it
    for i in range(it, max_iter):
        check = (i + 1) % n_iter_check == 0
        grad, kl = gradient(P, p, exaggeration)
        if check or i == max_iter - 1:
            error = kl
        inc = update * grad < 0.0
        gains[inc] += 0.2
        gains[~inc] *= 0.8
        np.clip(gains, 0.01, np.inf, out=gains)
        grad *= gains
        update = momentum * update - lr * grad
        p = p + update
        if check:
            if error < best_error:
                best_error, best_iter = error, i
            elif i - best_iter > n_iter_without_progress:
                break
            if np.linalg.norm(grad) <= min_grad_norm:
                break
    return p, error, i


def fit(D, perplexity=30.0, early_exaggeration=12.0, max_iter=1000, n_iter_without_progress=300, min_grad_norm=1e-7,
        random_state=0, init=None):
    """{"embedding", "kl_divergence", "n_iter", "learning_rate", "P"} of the whole fit."""
    n = np.asarray(D).shape[0]
    P = joint_probabilities(D, perplexity)
    lr = np.maximum(n / early_exaggeration / 4, 50)
    Y = (random_init(n, random_state) if init is None else np.asarray(init)).astype(np.float64)
    Y, kl, it = _descend(P, Y, 0, 250, 0.5, lr, early_exaggeration, 250, min_grad_norm)
    if it < 250 or max_iter - 250 > 0:
        Y, kl, it = _descend(P, Y, it + 1, max_iter, 0.8, lr, 1.0, n_iter_without_progress, min_grad_norm)
    return {"embedding": Y, "kl_divergence": kl, "n_iter": it, "learning_rate": lr, "P": P}
