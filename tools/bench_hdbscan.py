#!/usr/bin/env python3
"""Time phyloselect's HDBSCAN on the matrix resident after the distance stage, at C2's shape (100 000
contigs x 20 kb, fixed-length synthetic FASTA generated on the device, k=4 both strands, JSD, float32):
the input check, the core distances, every Boruvka round (components left, GB/s of its one pass over the
matrix against the HBM figure bench.py's select leg uses), the host stage and the whole fit, for
min_cluster_size 5 and 50.  For comparison, scikit-learn's HDBSCAN on the CPU on a 20 000-row sample of the
same matrix.  Prints one JSON document (and writes it to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from phyloligo_b200 import engine, phyloselect, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def hbm_figure():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
    except (OSError, ValueError):
        return 6650.0


def event_ms(fn, reps=3):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def stages(D, mcs, hbm):
    n = int(D.shape[0])
    nbytes = n * n * D.element_size()
    out = {"min_cluster_size": mcs, "min_samples": mcs}
    out["check_ms"] = event_ms(lambda: phyloselect.check_matrix(D))
    out["check_gbs"] = nbytes / (out["check_ms"] * 1e-3) / 1e9
    out["core_ms"] = event_ms(lambda: phyloselect.kth_smallest(D, mcs + 1))
    out["core_note"] = "exact radix select: %d histogram passes over every row" % D.element_size()
    core = phyloselect.kth_smallest(D, mcs + 1)
    phyloselect.mutual_reachability_mst(D, core)  # warm-up
    torch.cuda.synchronize()
    marks = [torch.cuda.Event(enable_timing=True)]
    comps = []

    def on_round(c):
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        marks.append(ev)
        comps.append(c)

    marks[0].record()
    u, v, w = phyloselect.mutual_reachability_mst(D, core, on_round)
    torch.cuda.synchronize()
    rounds = []
    for r, c in enumerate(comps):
        ms = marks[r].elapsed_time(marks[r + 1])
        gbs = nbytes / (ms * 1e-3) / 1e9
        rounds.append({"round": r + 1, "ms": ms, "components_after": c, "gbs": gbs, "frac_of_hbm": gbs / hbm})
    out["boruvka_rounds"] = rounds
    out["mst_ms"] = sum(r["ms"] for r in rounds)
    uh, vh, wh = u.cpu().numpy(), v.cpu().numpy(), w.cpu().numpy().astype(np.float64)
    t0 = time.perf_counter()
    labels = phyloselect.hdbscan_tree(uh, vh, wh, n, mcs)[0]
    out["host_stage_ms"] = (time.perf_counter() - t0) * 1e3
    h = phyloselect.HDBSCAN(min_cluster_size=mcs)
    h.fit(D)  # warm-up of the whole path
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    h.fit(D)
    torch.cuda.synchronize()
    out["total_ms"] = (time.perf_counter() - t0) * 1e3
    out["clusters"] = int(h.labels_.max() + 1)
    out["noise"] = int((h.labels_ == -1).sum())
    assert np.array_equal(h.labels_, labels)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--length", type=int, default=20_000)
    ap.add_argument("--sample", type=int, default=20_000, help="rows of the scikit-learn comparison (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = engine.require_cuda()
    hbm = hbm_figure()
    doc = {"card": card(), "hbm_figure_gbs": hbm,
           "workload": "%d contigs x %d bp (synth.device_fasta, seed 2), k=4 both strands, JSD float32 matrix resident (%.1f GB)"
                       % (args.n, args.length, args.n * args.n * 4 / 1e9)}
    text, b, e, _ = synth.device_fasta(args.n, args.length, 2, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    del text
    D = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    torch.cuda.synchronize()
    doc["runs"] = [stages(D, mcs, hbm) for mcs in (5, 50)]
    if args.sample:
        m = min(args.sample, args.n)
        rows = np.sort(np.random.default_rng(0).choice(args.n, m, replace=False))
        idx = torch.from_numpy(rows).to(dev)
        S = D.index_select(0, idx).index_select(1, idx).contiguous()
        Sh = S.cpu().numpy().astype(np.float64)
        from sklearn.cluster import HDBSCAN as SkHDBSCAN
        t0 = time.perf_counter()
        sk = SkHDBSCAN(min_cluster_size=5, min_samples=6, metric="precomputed", copy=True).fit(Sh)
        sk_s = time.perf_counter() - t0
        h = phyloselect.HDBSCAN(min_cluster_size=5)
        h.fit(S)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        h.fit(S)
        torch.cuda.synchronize()
        dev_s = time.perf_counter() - t0
        doc["sample"] = {"rows": m, "how": "rows and columns of the matrix at %d seeded random indices (seed 0), float64 for "
                                           "scikit-learn" % m,
                         "sklearn_cpu_s": sk_s, "sklearn_clusters": int(sk.labels_.max() + 1),
                         "device_s": dev_s, "device_clusters": int(h.labels_.max() + 1), "cpu_threads": os.cpu_count()}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
