"""CPU tests: the oracle restatement against the reference's own outputs.

The golden vectors were produced by tests/golden/make_golden.py, which executes
the reference's function bodies (bin/phyloligo.py:601-661, core/phylodist.py:12-68)
AST-extracted from the reference's sources.
"""
import math

import numpy as np
import pytest
import scipy.spatial.distance as ssd
import scipy.stats as sst

from conftest import golden_case_arrays
from oracle import phylo_oracle as po
from phyloligo_b200 import synth


def test_profile_oracle_matches_reference_golden(profile_golden):
    seqs = profile_golden["sequences"]
    assert len(profile_golden["cases"]) > 500
    for case in profile_golden["cases"]:
        counts, total, freq = golden_case_arrays(case)
        seq, pat, strand = seqs[case["seq"]], case["pattern"], case["strand"]
        c_lit, t_lit = po.count_vector(seq, pat, strand)
        assert t_lit == total
        assert np.array_equal(c_lit, counts)
        c_np, t_np = po.count_vector_np(seq, pat, strand)
        assert t_np == total
        assert np.array_equal(c_np, counts)
        f = po.compute_frequency(seq, pat, strand)
        assert np.array_equal(np.asarray(f, dtype=np.float64), freq)  # bit exact
        assert np.array_equal(po.frequency_np(seq, pat, strand), freq)


def test_known_answers():
    # SURVEY.md section 4 known-answer vectors (derived from the reference bodies)
    words, total = po.cut_sequence_and_count_pattern("ACGTNACGTA", "101")
    assert dict(words) == {"AG": 2, "CT": 2, "GA": 1} and total == 5
    assert po.select_strand("AACG", "both") == "AACGCGTT"
    words, total = po.cut_sequence_and_count_pattern("AACGCGTT", "11")
    assert dict(words) == {"AA": 1, "AC": 1, "CG": 2, "GC": 1, "GT": 1, "TT": 1} and total == 7
    order = ["".join(p) for p in __import__("itertools").product(po.ALPHABET, repeat=2)]
    assert order == "CC CG CA CT GC GG GA GT AC AG AA AT TC TG TA TT".split()
    a = np.array([0.25, 0.25, 0.5, 0.0])
    assert po.JSD(a, a) == 0.0
    e0, e1 = np.eye(4)[0], np.eye(4)[1]
    assert po.JSD(e0, e1) == 0.6931471805599453
    f = po.compute_frequency("", "1111", "both")
    assert f.shape == (256,) and not f.any() and f.dtype.kind == "i"
    z = np.zeros(4)
    assert abs(po.JSD(z, a) - 0.5 * math.log(2)) < 1e-15 and po.JSD(z, z) == 0.0


def test_distance_oracle_matches_reference_golden(distance_golden):
    for name in ("real_k4", "sparse_64", "onehot_16"):
        X = distance_golden[name + "_X"]
        n = X.shape[0]
        for a in range(n):
            for b in range(n):
                assert po.Eucl(X[a], X[b]) == distance_golden[name + "_Eucl"][a, b]
                assert po.JSD(X[a], X[b]) == distance_golden[name + "_JSD"][a, b]
        X32 = X.astype(np.float32)
        j2 = po.JSD(X32, X32[: max(2, n // 2)])
        assert j2.dtype == np.float32
        assert np.array_equal(j2, distance_golden[name + "_JSD2d_f32"])
        # vectorised oracle agrees with the pair functions
        assert np.allclose(po.pairwise_np(X, "JSD"), distance_golden[name + "_JSD"], rtol=1e-12, atol=1e-15)
        assert np.allclose(po.pairwise_np(X, "Eucl"), distance_golden[name + "_Eucl"], rtol=1e-12, atol=1e-15)


def test_reverse_complement_iupac():
    assert po.reverse_complement("ACGTN") == "NACGT"
    assert po.reverse_complement("acgtRYKM") == "KMRYacgt"
    assert po.reverse_complement("A-C*G") == "C*G-T"


def test_bc_kt_sc_against_scipy():
    rng = np.random.default_rng(11)
    for trial in range(40):
        d = int(rng.integers(2, 40))
        a = rng.integers(0, 4, d).astype(np.float64)  # tie heavy
        b = rng.integers(0, 4, d).astype(np.float64)
        if trial % 5 == 0:
            a = rng.random(d)
            b = rng.random(d)
        if (a + b).sum() > 0:
            assert po.BC(a, b) == pytest.approx(ssd.braycurtis(a, b), rel=1e-14, abs=1e-300)
        tau = sst.kendalltau(a, b).statistic
        kt = po.KT(a, b)
        assert kt == pytest.approx(1.0 - po.kendall_distance(a, b), abs=1e-15)
        if np.isnan(tau):
            assert kt == 0.0  # Bio.Cluster: constant row -> distance 1
        else:
            assert kt == pytest.approx(tau, abs=1e-12)
        rho = sst.spearmanr(a, b).statistic
        sc = po.SC(a, b)
        if np.isnan(rho):
            assert np.isnan(sc)
        else:
            assert sc == pytest.approx(1.0 - rho, abs=1e-12)
        assert np.array_equal(po.rank_average(a), sst.rankdata(a))
    assert po.KT(np.ones(5), np.arange(5.0)) == 0.0
    assert po.kendall_distance([1.0], [2.0]) == 0.0


def test_profile_properties():
    # (i) both = plus + minus + junction, (ii) total = sum over valid runs of (len - P + 1)
    import re
    for s in synth.make_sequences(5, 600, seed=9):
        s = s.decode()
        for pat in ("1111", "10101", "111010011"):
            cp, tp = po.count_vector_np(s, pat, "plus")
            cm, tm = po.count_vector_np(s, pat, "minus")
            cb, tb = po.count_vector_np(s, pat, "both")
            P = len(pat)
            runs = [len(r) for r in re.split("[^ACGT]+", s.upper()) if len(r) >= P]
            assert tp == tm == sum(r - P + 1 for r in runs)
            junction = cb - cp - cm
            assert (junction >= 0).all() and junction.sum() <= P - 1


def test_kount_oracle_replays_the_reference_goldens(tmp_path):
    """oracle/kount_oracle.py against outputs of the reference's own Kount.py function bodies
    (tests/golden/make_kount_golden.py): window coordinates exact, distances to 1e-12."""
    import json
    import os

    from oracle import kount_oracle as ko

    cases = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "kount_golden.json")))
    assert len(cases) >= 4
    for ci, case in enumerate(cases):
        path = os.path.join(tmp_path, "asm%d.fasta" % ci)
        with open(path, "w") as fh:
            fh.write(case["fasta"])
        records = ko.read_records(path)
        mcp = ko.compute_whole_composition(records, case["pattern"], case["strand"])
        want_mcp = np.array([float.fromhex(v) for v in case["mcp"]])
        assert np.array_equal(mcp, want_mcp)
        for dist, rows in case["rows"].items():
            got = ko.sliding_windows_distances(records, mcp, dist, case["pattern"], case["window"], case["step"],
                                               case["strand"], case["n_max"])
            assert [r[:3] for r in got] == [r[:3] for r in rows]
            g = np.array([r[3] for r in got])
            w = np.array([float.fromhex(r[3]) for r in rows])
            assert np.allclose(g, w, rtol=1e-12, atol=1e-15), (dist, np.abs(g - w).max())
