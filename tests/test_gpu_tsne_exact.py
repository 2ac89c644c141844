"""phyloselect's t-SNE (csrc/po_tsne.cu) held to exact references: whole fits bit for bit against scikit-learn's own
_gradient_descent driven through the device gradient, single optimiser steps from crafted state against numpy in
scikit-learn's dtypes, the repulsion pass at every change of its launch geometry up to C2's 100 000 rows against a
float64 all-pairs sum, and the affinities at the perplexity search's register-slot edges."""
import numpy as np
import pytest
import torch
from scipy.sparse import csr_matrix

from oracle import tsne_oracle as to
from phyloligo_b200 import phyloselect
from test_hdbscan_oracle import blobs, jsd_matrix
from test_tsne_oracle import sklearn_descent, sklearn_P

pytestmark = pytest.mark.gpu

# the repulsion launch geometry of po_tsne.cu
REP_ROWS, REP_TILE, REP_TARGET_CTAS = 512, 256, 4096


# ---------------------------------------------------------------------------------------------------------------
# A. whole fits, bit for bit, against scikit-learn's TSNE._tsne with the device as its objective
# ---------------------------------------------------------------------------------------------------------------
FITS = [  # id, n, perplexity, matrix, TSNE arguments
    ("auto", 600, 30.0, "blobs", {}),
    ("lr200", 600, 30.0, "blobs", {"learning_rate": 200.0}),
    ("ee7", 600, 30.0, "blobs", {"early_exaggeration": 7.0}),
    ("ee7-lr200", 600, 30.0, "blobs", {"early_exaggeration": 7.0, "learning_rate": 200.0}),
    ("max250", 600, 30.0, "blobs", {"max_iter": 250}),
    ("max251-lr200", 600, 30.0, "blobs", {"max_iter": 251, "learning_rate": 200.0}),
    ("max300", 600, 30.0, "blobs", {"max_iter": 300}),
    ("min-grad-norm", 600, 30.0, "blobs", {"min_grad_norm": 1e3}),
    ("no-progress", 120, 20.0, "jsd", {"n_iter_without_progress": 0}),
    ("n2", 2, 1.5, "blobs", {}),
    ("n9", 9, 2.0, "blobs", {"learning_rate": 200.0}),
    ("n1500", 1500, 30.0, "blobs", {"early_exaggeration": 7.0}),
    ("n1500-lr200", 1500, 50.0, "jsd", {"learning_rate": 200.0}),
]


class _Recording(phyloselect._Descent):
    """_Descent that keeps the positions entering every 50th gradient evaluation (iteration 0, 50, ...)."""
    seen = None

    def gradient(self, *args, **kwargs):
        self.calls = getattr(self, "calls", 0)
        if self.calls % 50 == 0:
            _Recording.seen[self.calls] = self.Y.cpu().numpy()
        self.calls += 1
        return super().gradient(*args, **kwargs)


@pytest.mark.parametrize("name,n,perplexity,kind,kwargs", FITS, ids=[f[0] for f in FITS])
def test_fit_equals_scikit_learns_descent_bit_for_bit(monkeypatch, name, n, perplexity, kind, kwargs):
    D = blobs(n, 5) if kind == "blobs" else jsd_matrix(n, 3)
    Y0 = to.random_init(n, 11)
    P = phyloselect.tsne_affinities(D, perplexity, as_sparse=True)
    ee = kwargs.get("early_exaggeration", 12.0)
    stage2 = P.data * ee * (1.0 / ee)  # what scipy's P *= ee, P /= ee leaves
    if ee != 12.0:
        assert (stage2 != P.data).any()
    dev = torch.device("cuda")
    st = phyloselect._Descent(phyloselect._device_csr(P, dev), Y0)
    grad = torch.empty((n, 2), dtype=torch.float32, device=dev)
    sk_seen = {}

    def objective(Pk, params, compute_error):  # _kl_divergence_bh on the device, on the P scikit-learn has scaled
        calls = len(objective.calls)
        objective.calls.append(compute_error)
        if calls % 50 == 0:
            sk_seen[calls] = params.reshape(n, 2).copy()
        st.P[2].copy_(torch.from_numpy(Pk.data))
        st.Y.copy_(torch.from_numpy(params.reshape(n, 2)))
        kl, _ = st.gradient(1.0, 1.0, grad=grad, compute_error=compute_error)
        return (kl if compute_error else np.nan), grad.cpu().numpy().ravel()

    objective.calls = []
    Y, kl, n_iter = sklearn_descent(monkeypatch, P, Y0, objective, perplexity=perplexity, **kwargs)
    monkeypatch.undo()
    _Recording.seen = {}
    monkeypatch.setattr(phyloselect, "_Descent", _Recording)
    t = phyloselect.TSNE(init=Y0, perplexity=perplexity, **kwargs).fit(D)
    assert sorted(_Recording.seen) == sorted(sk_seen)
    for it in sorted(sk_seen):
        assert np.array_equal(_Recording.seen[it], sk_seen[it]), "positions differ entering iteration %d" % it
    assert t.embedding_.dtype == np.float32 and np.array_equal(t.embedding_, Y)
    assert t.kl_divergence_ == kl and t.n_iter_ == n_iter
    if name == "max250":  # _tsne still enters stage 2, which runs no step: n_iter_ 250 and the initial error
        assert n_iter == 250 and len(objective.calls) == 250 and kl == np.finfo(float).max
        return
    assert len(objective.calls) == n_iter + 1 and objective.calls[-1]
    if name == "min-grad-norm":
        assert n_iter == 99  # both stages stop at their first check
    elif name == "no-progress":
        assert n_iter < 999
    elif n >= 600:
        assert n_iter == kwargs.get("max_iter", 1000) - 1


# ---------------------------------------------------------------------------------------------------------------
# B. one optimiser step from crafted state against numpy in scikit-learn's dtypes
# ---------------------------------------------------------------------------------------------------------------
def random_P(n, k, seed):
    """A symmetric CSR P: k random neighbours per row (never the row itself), summed with its transpose, total 1."""
    rng = np.random.default_rng(seed)
    cols = rng.integers(0, n - 1, size=(n, k))
    cols += cols >= np.arange(n)[:, None]
    C = csr_matrix((rng.random(n * k), cols.ravel(), np.arange(0, n * k + 1, k)), shape=(n, n))
    P = (C + C.T).tocsr()
    P.sum_duplicates()
    P.sort_indices()
    P.data /= P.data.sum()
    return P


def numpy_step(Y, g, update, gains, momentum, lr):
    """_gradient_descent's step with its dtypes: update float64 or float32, gains and positions float32."""
    update, gains, p = update.copy(), gains.copy(), Y.ravel().copy()
    inc = update * g < 0.0
    gains[inc] += 0.2
    gains[~inc] *= 0.8
    np.clip(gains, 0.01, np.inf, out=gains)
    g = g * gains
    update = momentum * update - lr * g
    p += update
    return p.reshape(-1, 2), update, gains, np.dot(g.astype(np.float64), g.astype(np.float64))


@pytest.mark.parametrize("update64", [True, False], ids=["float64-update", "float32-update"])
@pytest.mark.parametrize("momentum", [0.5, 0.8])
def test_one_step_from_crafted_state(update64, momentum):
    n = 256
    rng = np.random.default_rng(7)
    Y = rng.normal(0, 2, size=(n, 2)).astype(np.float32)
    Y[-1] = 1e15  # so far out that its q^2 underflows: a row with gradient +0 (it has no P entries)
    P = random_P(n - 1, 5, 3)
    P = csr_matrix((P.data, P.indices, np.append(P.indptr, P.indptr[-1])), shape=(n, n))
    dev = torch.device("cuda")
    st = phyloselect._Descent(phyloselect._device_csr(P, dev), Y)
    grad = torch.empty((n, 2), dtype=torch.float32, device=dev)
    st.gradient(1.0, 1.0, grad=grad)
    g = grad.cpu().numpy().ravel()
    assert (g[-2:] == 0).all() and (g[:-2] != 0).all()
    # crafted state, one pattern per element (cycled): the first iteration's zero update, both signs of update * g,
    # gains at, just above and just below the clip, and in float32 an update * g that is subnormal and negative
    m = 2 * n
    ftype = np.float64 if update64 else np.float32
    s = np.sign(g).astype(ftype)
    s[s == 0] = 1
    kind = np.arange(m) % 6
    update = np.where(kind == 0, 0.0, np.where(kind % 2 == 1, -s, s) * np.exp(rng.normal(0, 3, m))).astype(ftype)
    sub = (kind == 5) & (g != 0)
    update[sub] = (-s[sub] * np.float32(1e-40) / np.abs(g[sub])).astype(ftype)
    if not update64:
        prod = update[sub] * g[sub]
        assert (prod < 0).all() and (np.abs(prod) < np.finfo(np.float32).tiny).all()  # subnormal, not flushed
    gains = np.choose(np.arange(m) % 5, [np.float32(0.01), np.nextafter(np.float32(0.01), np.float32(1)),
                                         np.float32(0.0125), np.float32(0.012), np.float32(1.7)]).astype(np.float32)
    gains *= np.where(np.arange(m) % 7 == 0, np.float32(3.0), np.float32(1.0))
    lr = np.float64(123.45678) if update64 else 200.0
    st.update.copy_(torch.from_numpy(update.astype(np.float64).reshape(n, 2)))
    st.gains.copy_(torch.from_numpy(gains.reshape(n, 2)))
    grad2 = torch.empty_like(grad)
    _, gn2 = st.gradient(1.0, 1.0, Y_next=st.Y_next, grad=grad2, momentum=momentum, lr=lr, update64=update64,
                         compute_error=True)
    assert np.array_equal(grad2.cpu().numpy().ravel(), g)
    want_Y, want_update, want_gains, want_gn2 = numpy_step(Y, g, update, gains, momentum, lr)
    assert want_update.dtype == ftype
    assert np.array_equal(st.Y_next.cpu().numpy(), want_Y)
    assert np.array_equal(st.update.cpu().numpy().ravel(), want_update.astype(np.float64))
    assert np.array_equal(st.gains.cpu().numpy().ravel(), want_gains)
    assert gn2 == pytest.approx(want_gn2, rel=1e-12)


def test_second_stage_probabilities_are_scipys_reciprocal_scaling():
    # scipy's P /= ee multiplies by 1.0 / ee; entries one float64 step below a float32 rounding midpoint tell that
    # apart from a division.  The device, scaling P by (mul, div), must read the float32 bits of the data _tsne leaves.
    ee = 10.0
    rng = np.random.default_rng(2)
    f = (rng.random(20000) * 1e-3).astype(np.float32)
    mid = (f.astype(np.float64) + np.nextafter(f, np.float32(1)).astype(np.float64)) / 2
    p = mid - np.spacing(mid)
    hits = p[(p * ee * (1.0 / ee)).astype(np.float32) != (p * ee / ee).astype(np.float32)]
    assert hits.size >= 64
    n = 128
    P = random_P(n, 4, 9)
    P.data[:64] = hits[:64]
    P.data[64:] = 1e-3
    Y = rng.normal(0, 1, size=(n, 2)).astype(np.float32)
    scaled = P.copy()
    scaled *= ee
    scaled /= ee
    dev = torch.device("cuda")
    g_dev, g_want = (torch.empty((n, 2), dtype=torch.float32, device=dev) for _ in range(2))
    kl_dev, _ = phyloselect._Descent(phyloselect._device_csr(P, dev), Y).gradient(ee, ee, grad=g_dev, compute_error=True)
    kl_want, _ = phyloselect._Descent(phyloselect._device_csr(scaled, dev), Y).gradient(1.0, 1.0, grad=g_want,
                                                                                          compute_error=True)
    assert kl_dev == kl_want and torch.equal(g_dev, g_want)


# ---------------------------------------------------------------------------------------------------------------
# C. repulsion and gradient at every geometry boundary, against a float64 all-pairs sum on the device
# ---------------------------------------------------------------------------------------------------------------
def geometry(n):
    """(row CTAs, tiles, chunks, tiles per chunk, empty chunks) of po_tsne_repulsion for n rows."""
    row_ctas, tiles = -(-n // REP_ROWS), -(-n // REP_TILE)
    chunks = min(max(-(-REP_TARGET_CTAS // row_ctas), 1), tiles)
    per = -(-tiles // chunks)
    return row_ctas, tiles, chunks, per, chunks - -(-n // (per * REP_TILE))


def exact_gradient(P, Y, exaggeration=1.0, chunk=1024):
    """float64 on the device: (grad [n, 2], KL, Z, per-row force scale 4 (sum |attraction terms| + sum |repulsion
    terms| / Z)) for P * exaggeration read as float32, every pair summed exactly."""
    dev = torch.device("cuda")
    Yd = torch.from_numpy(np.asarray(Y, dtype=np.float32)).to(dev).double()
    n = Yd.shape[0]
    rep = torch.zeros((n, 2), dtype=torch.float64, device=dev)
    rep_abs = torch.zeros(n, dtype=torch.float64, device=dev)
    Z = torch.zeros((), dtype=torch.float64, device=dev)
    for r0 in range(0, n, chunk):
        r1 = min(n, r0 + chunk)
        dx = Yd[r0:r1, 0, None] - Yd[None, :, 0]
        dy = Yd[r0:r1, 1, None] - Yd[None, :, 1]
        d2 = dx * dx + dy * dy
        q = 1.0 / (1.0 + d2)
        q[torch.arange(r1 - r0, device=dev), torch.arange(r0, r1, device=dev)] = 0.0
        Z += q.sum()
        q2 = q * q
        rep[r0:r1, 0] = (q2 * dx).sum(1)
        rep[r0:r1, 1] = (q2 * dy).sum(1)
        rep_abs[r0:r1] = (q2 * d2.sqrt()).sum(1)
        del dx, dy, d2, q, q2
    indptr = torch.from_numpy(np.asarray(P.indptr, dtype=np.int64)).to(dev)
    cols = torch.from_numpy(np.asarray(P.indices, dtype=np.int64)).to(dev)
    rows = torch.repeat_interleave(torch.arange(n, device=dev), indptr[1:] - indptr[:-1])
    p32 = torch.from_numpy((P.data * exaggeration).astype(np.float32)).to(dev).double()
    b = Yd[rows] - Yd[cols]
    qa = 1.0 / (1.0 + (b * b).sum(1))
    att = torch.zeros((n, 2), dtype=torch.float64, device=dev).index_add_(0, rows, (p32 * qa)[:, None] * b)
    att_abs = torch.zeros(n, dtype=torch.float64, device=dev).index_add_(0, rows, p32 * qa * b.norm(dim=1))
    tiny = float(np.finfo(np.float32).tiny)
    kl = (p32 * torch.log(p32.clamp(min=tiny) / (qa / Z).clamp(min=tiny))).sum()
    g = 4.0 * (att - rep / Z)
    return g.cpu().numpy(), float(kl), float(Z), (4.0 * (att_abs + rep_abs / Z)).cpu().numpy()


def device_gradient(P, Y, exaggeration=1.0):
    """(grad, KL, Z) of the device, its workspace filled with NaN beforehand so no partial it leaves unwritten
    can pass unseen."""
    dev = torch.device("cuda")
    st = phyloselect._Descent(phyloselect._device_csr(P, dev), Y)
    st.work.fill_(0xFF)
    grad = torch.empty((st.n, 2), dtype=torch.float32, device=dev)
    kl, _ = st.gradient(exaggeration, 1.0, grad=grad, compute_error=True)
    n, chunks = st.n, geometry(st.n)[2]
    Z = float(st.work.view(torch.float64)[3 * chunks * n + 5 * n])  # the workspace's sums[0]
    return grad.cpu().numpy(), kl, Z


def positions(kind, n, seed):
    rng = np.random.default_rng(seed)
    if kind == "coincident":  # a third of the rows duplicate others, and a block sits on one point
        Y = rng.normal(0, 1, size=(n, 2)).astype(np.float32)
        Y[: n // 3] = Y[rng.integers(n // 3, n, n // 3)]
        Y[n // 3: n // 3 + min(40, n // 4)] = Y[n - 1]
        return Y
    return rng.normal(0, {"scale3": 3.0, "scale1e-4": 1e-4}[kind], size=(n, 2)).astype(np.float32)


ROW_TOL = 3e-7  # of the row's force scale; at most 1.0e-7 measured on a B200
GEOMETRY_NS = [2, 3, 31, 33, 255, 256, 257, 511, 512, 513, 1025, 4097, 23040, 23041, 30000, 50000, 100000]


def check_gradient(P, Y, exaggeration=1.0):
    g, kl, Z = device_gradient(P, Y, exaggeration)
    g_ref, kl_ref, Z_ref, scale = exact_gradient(P, Y, exaggeration)
    assert np.isfinite(g).all()
    err = np.abs(g.astype(np.float64) - g_ref).max(1)
    row = (err / np.maximum(scale, 1e-300)).max()
    print("n %d: max row error %.3g of the force scale, %.3g of max|g|; KL error %.3g, Z %.3g relative" % (
        len(Y), row, err.max() / np.abs(g_ref).max(), abs(kl - kl_ref), abs(Z - Z_ref) / Z_ref))
    # po_tsne_repulsion adds each row's own q_ii = 1 into its float32 Z run and removes it in float64, which costs
    # up to 2^-24 per row of Z: n 2^-24 / Z of the repulsion, seen only when Z is small (n = 2 at scale 3)
    assert (err <= (ROW_TOL + len(Y) * 2.0 ** -24 / Z_ref) * scale).all(), "row error %.3g of its force scale" % row
    # the KL terms read q_ij in float32, as scikit-learn does: up to 2^-24 of log-error per unit of p, which shows
    # where the KL itself is near 0 (a few points at the 1e-4 init scale)
    # (the q_ii loss above adds n 2^-24 / Z to log Z)
    z_loss = len(Y) * 2.0 ** -24
    assert abs(kl - kl_ref) <= 1e-6 * abs(kl_ref) + (2.0 ** -23 + z_loss / Z_ref) * exaggeration * P.data.sum()
    assert abs(Z - Z_ref) <= 1e-6 * Z_ref + z_loss
    return g, g_ref


def test_exact_reference_equals_the_oracle():
    for n in (3, 257, 700):
        P = random_P(n, min(n - 1, 6), n)
        for kind in ("scale3", "scale1e-4", "coincident"):
            Y = positions(kind, n, 1)
            for ex in (1.0, 12.0):
                g, kl, _, _ = exact_gradient(P, Y, ex, chunk=100)
                g_or, kl_or = to.gradient(P, Y, ex)
                assert np.abs(g - g_or).max() <= 1e-12 * np.abs(g_or).max() and kl == pytest.approx(kl_or, rel=1e-12)


def test_geometry_reaches_every_boundary():
    assert geometry(20000) == (40, 79, 79, 1, 0)
    assert geometry(23040) == (45, 90, 90, 1, 0)
    assert geometry(23041) == (46, 91, 90, 2, 44)
    assert geometry(30000) == (59, 118, 70, 2, 11)
    assert geometry(50000) == (98, 196, 42, 5, 2)
    assert geometry(100000) == (196, 391, 21, 19, 0)
    lib = phyloselect._lib.load()
    for n in GEOMETRY_NS:  # the workspace holds 3 float64 partials per chunk and row: the library's chunk count
        assert lib.po_tsne_workspace(n) == (3 * geometry(n)[2] * n + 5 * n + 4) * 8


@pytest.mark.parametrize("n", GEOMETRY_NS)
def test_gradient_at_every_geometry_boundary(n):
    P = random_P(n, min(n - 1, 8), n)
    kinds = ("scale3", "scale1e-4", "coincident") if n <= 23041 else ("scale3", "scale1e-4")
    for kind in kinds:
        for ex in ((1.0, 12.0) if n <= 4097 else (1.0,)):
            check_gradient(P, positions(kind, n, n + 1), ex)


GLOBAL_TOL = 8e-5  # of max|g| at converged positions


@pytest.mark.parametrize("n", [500, 3000])
def test_gradient_at_converged_positions(n):
    """Near convergence attraction and repulsion cancel to a few digits, so the repulsion's rounding shows in the
    gradient.  Measured on a B200: the two float32 levels of po_tsne_repulsion keep it to 4.5e-5 of max|g| at
    n = 500 (1.6e-5 at 3000), where one flat float32 run per tile gives 1.3e-4 (2.3e-5); scikit-learn's own
    float32 gradient is 2.8e-4 away at n = 500."""
    D = blobs(n, 4)
    P = phyloselect.tsne_affinities(D, 30.0, as_sparse=True)
    Y = phyloselect.TSNE(random_state=1).fit(D).embedding_
    g, g_ref = check_gradient(P, Y)
    rel = np.abs(g - g_ref).max() / np.abs(g_ref).max()
    assert rel <= GLOBAL_TOL, "%.3g of max|g|" % rel


# ---------------------------------------------------------------------------------------------------------------
# D. affinities at the register-slot edges of po_tsne_conditional (32 neighbours per slot, 32 slots)
# ---------------------------------------------------------------------------------------------------------------
def check_affinities(D, perplexity, with_sklearn=True):
    """Structure equal to the oracle's and scikit-learn's, every value within 1e-9 of one of them: the two differ
    by up to a few 1e-9 where a row's entropy lands on the search's tolerance and their sum orders stop the search a
    step apart."""
    got = phyloselect.tsne_affinities(torch.from_numpy(np.ascontiguousarray(D)).cuda(), perplexity, as_sparse=True)
    err = None
    for want in (to.joint_probabilities(D, perplexity),) + ((sklearn_P(D, perplexity),) if with_sklearn else ()):
        assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
        e = np.abs(got.data - want.data)
        err = e if err is None else np.minimum(err, e)
    assert err.max() <= 1e-9


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("k,perplexity", [(31, 10.0), (32, 10.34), (33, 10.67), (64, 21.0), (65, 21.34), (1024, 341.0)])
def test_affinities_at_register_slot_edges(k, perplexity, dtype):
    assert int(3.0 * perplexity + 1) == k
    n = 1100 if k == 1024 else 400
    check_affinities(blobs(n, k).astype(dtype), perplexity)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("shape", ["duplicate-rows", "underflow"])
def test_affinities_of_degenerate_matrices(shape, dtype):
    D = np.array(blobs(300, 12))
    if shape == "duplicate-rows":  # zero distances between a row and its copy
        src = np.arange(0, 300, 3)
        X = np.arange(300)
        X[src + 1] = src
        D = D[X][:, X]
        np.fill_diagonal(D, 0.0)
    else:  # every exp(-d^2 beta) underflows at beta = 1: the search starts from sum_p = 1e-8
        off = ~np.eye(300, dtype=bool)
        D = D * (40.0 / D[off].min())
        assert (np.exp(-(D[off].astype(dtype) ** 2).astype(np.float32).astype(np.float64)) == 0).all()
    # a row's copies tie with each other in every other row; scikit-learn orders exact ties its own way, the
    # device and the oracle by column (stable sort)
    check_affinities(D.astype(dtype), 30.0, with_sklearn=shape != "duplicate-rows")
