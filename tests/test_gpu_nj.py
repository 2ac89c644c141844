"""GPU parity of phyloselect's neighbour-joining trees (phyloligo_b200/phyloselect.py: nj, write_nj_newick,
--tree-method; csrc/po_nj.cu) against oracle/nj_oracle.py, bit for bit."""
import os

import numpy as np
import pytest
import torch

from oracle import nj_oracle
from phyloligo_b200 import _lib, engine, phyloselect, synth
from phyloligo_b200._lib import PhyloligoError
from test_gpu_linkage import kt_style, quantised
from test_hdbscan_oracle import blobs, jsd_matrix
from test_nj_oracle import TEXTBOOK, random_tree, tree_splits

pytestmark = pytest.mark.gpu

METHODS = list(phyloselect.NJ_METHODS)


def assert_same(D, method):
    want_e, want_l = nj_oracle.nj(D, method)
    got_e, got_l = phyloselect.nj(D, method)
    assert np.array_equal(got_e, want_e)
    assert np.array_equal(got_l.view(np.uint64), want_l.view(np.uint64))


@pytest.mark.parametrize("method", METHODS)
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("make,n", [(blobs, 1500), (quantised, 1000), (kt_style, 800), (jsd_matrix, 600)])
def test_equals_oracle_bit_for_bit(make, n, dtype, method):
    D = make(n, 5).astype(dtype)
    assert_same(D, method)


@pytest.mark.parametrize("method", METHODS)
def test_small_matrices_and_ties(method):
    assert_same(TEXTBOOK, method)
    assert_same(np.array([[0.0, 3.0, 4.0], [3.0, 0.0, 5.0], [4.0, 5.0, 0.0]]), method)
    tie = np.array([[0, 8, 6, 3], [8, 0, 4, 9], [6, 4, 0, 7], [3, 9, 7, 0]], dtype=np.float64)
    assert_same(tie, method)
    p = [1, 0, 2, 3]
    assert_same(tie[np.ix_(p, p)], method)
    for n in (3, 4, 5, 40):
        assert_same(np.ones((n, n)) - np.eye(n), method)  # every Q ties at every join
        assert_same(np.zeros((n, n)), method)


@pytest.mark.parametrize("method", METHODS)
def test_additive_tree_recovered_at_eight_thousand_rows(method):
    n = 8000
    D, want = random_tree(n, 21)
    edge, length = phyloselect.nj(D, method)
    got = tree_splits(edge, length, n)
    assert set(got) == set(want)  # Robinson-Foulds distance 0
    assert max(abs(got[k] - want[k]) for k in want) <= 1e-9


@pytest.mark.parametrize("method", METHODS)
def test_float32_equals_its_float64_widening(method):
    D = jsd_matrix(500, 7)
    e32, l32 = phyloselect.nj(D, method)
    e64, l64 = phyloselect.nj(D.astype(np.float64), method)
    assert np.array_equal(e32, e64) and np.array_equal(l32.view(np.uint64), l64.view(np.uint64))


def test_device_input_unchanged_and_runs_repeat():
    Dd = torch.from_numpy(jsd_matrix(700, 3)).cuda()
    before = Dd.clone()
    _lib.timing_enable(True)
    _lib.timing_reset()
    for method in METHODS:
        a = phyloselect.nj(Dd, method)
        b = phyloselect.nj(Dd, method)
        assert torch.equal(Dd.view(torch.int32), before.view(torch.int32))
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64)), method
    ms, launches = _lib.timing_read(3)
    _lib.timing_enable(False)
    assert launches == 4 and ms > 0.0


def test_compactions_happen():
    # 300 rows: the 256-slot front headroom runs out, so the live block is packed at least once
    _, _, compactions = phyloselect.nj_raw(torch.from_numpy(blobs(300, 2)).cuda(), "nj")
    assert compactions >= 1


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_refusals(dtype, monkeypatch):
    D = blobs(100, 1).astype(dtype)
    A = D.copy()
    A[7, 42] = np.nextafter(A[7, 42], dtype(10))
    with pytest.raises(PhyloligoError, match=r"not symmetric: entry \(7, 42\)"):
        phyloselect.nj(A)
    N = D.copy()
    N[63, 12] = N[12, 63] = np.nan
    with pytest.raises(PhyloligoError, match=r"entry \(12, 63\) is NaN"):
        phyloselect.nj(N, "bionj")
    inf = D.copy()
    inf[99, 98] = inf[98, 99] = np.inf
    with pytest.raises(PhyloligoError, match=r"entry \(98, 99\) is infinite"):
        phyloselect.nj(inf)
    with pytest.raises(ValueError, match="method"):
        phyloselect.nj(D, "upgma")
    with pytest.raises(ValueError, match="at least 3"):
        phyloselect.nj(D[:2, :2])
    with pytest.raises(PhyloligoError, match="square"):
        phyloselect.nj(D[:, :50])
    with pytest.raises(PhyloligoError, match="1e50"):
        phyloselect.nj(np.full((4, 4), -1e60) + np.diag(np.full(4, 1e60)))
    # a working state that does not fit is refused before anything is allocated
    allocated = torch.cuda.memory_allocated()
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (1 << 16, 1 << 40))
    memory_allocated = torch.cuda.memory_allocated
    monkeypatch.setattr(torch.cuda, "memory_reserved", lambda device=None: memory_allocated(device))  # no cached blocks
    for method in METHODS:
        with pytest.raises(PhyloligoError, match=r"needs %d bytes" % phyloselect.nj_bytes(100, method)):
            phyloselect.nj(torch.from_numpy(D).cuda(), method)
    assert torch.cuda.memory_allocated() <= allocated + D.nbytes + 4096


def _read_dir(path):
    return {f: open(os.path.join(path, f), "rb").read() for f in sorted(os.listdir(path))}


def test_command_line(tmp_path, capsys):
    seqs = synth.make_sequences(300, 3000, seed=9)
    fasta = os.path.join(tmp_path, "asm.fa")
    synth.write_fasta(fasta, seqs, line=70)
    from phyloligo_b200 import phyloligo
    res, _, _ = phyloligo._profile_file(fasta, "1111", "both", ("freq32",))
    D_dev = engine.distance_matrix_device(res["freq32"], "JSD", torch.float32, symmetric=True).cpu().numpy()
    ids = phyloselect.fasta_record_ids(fasta)
    base = os.path.join(tmp_path, "base")
    assert phyloselect.main(["--assembly", fasta, "-d", "JSD", "--pattern", "1111", "-m", "kmedoids", "-k", "3", "-o", base]) == 0
    for method in METHODS:
        edge, length = nj_oracle.nj(D_dev, method)
        want = os.path.join(tmp_path, "want_%s.nwk" % method)
        phyloselect.write_nj_newick(edge, length, ids, want)
        out = os.path.join(tmp_path, "out_" + method)
        tree = os.path.join(tmp_path, "got_%s.nwk" % method)
        assert phyloselect.main(["--assembly", fasta, "-d", "JSD", "--pattern", "1111", "-m", "kmedoids", "-k", "3", "-o", out,
                                 "--tree-method", method, "--tree-out", tree]) == 0
        assert open(tree, "rb").read() == open(want, "rb").read()
        assert _read_dir(out) == _read_dir(base)  # the cluster files do not depend on the tree
    # from a matrix file, leaves named by row index
    np.savetxt(os.path.join(tmp_path, "m.txt"), D_dev.astype(np.float64), delimiter="\t")
    M = np.loadtxt(os.path.join(tmp_path, "m.txt"))
    tree = os.path.join(tmp_path, "m.nwk")
    assert phyloselect.main(["-i", os.path.join(tmp_path, "m.txt"), "-m", "hclust", "-k", "3", "-o", os.path.join(tmp_path, "hc"),
                             "--tree-method", "bionj", "--tree-out", tree]) == 0
    edge, length = nj_oracle.nj(M, "bionj")
    phyloselect.write_nj_newick(edge, length, [str(i) for i in range(300)], os.path.join(tmp_path, "want_m.nwk"))
    assert open(tree, "rb").read() == open(os.path.join(tmp_path, "want_m.nwk"), "rb").read()
    capsys.readouterr()
