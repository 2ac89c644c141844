#!/usr/bin/env python3
"""Time phyloselect's hierarchical clustering on the matrix resident after the distance stage, at C2's shape
(100 000 contigs x 20 kb, fixed-length synthetic FASTA generated on the device, k=4 both strands, JSD, float32):
for every linkage method the whole fit (input check, working copy, the persistent launch, host stage, as
`fit_s`), linkage_raw (the same without the host stage, `linkage_raw_s`), the cooperative launch alone (CUDA events,
timing family 2, `launch_s`), its grid-barrier count and microseconds per phase of that launch, against the
barrier floor po_microbench kind 4 measures in the same run.  For comparison, scipy.cluster.hierarchy.linkage on the CPU on a 20 000-row sample of
the same matrix beside the device on that sample (the two results compared bit for bit).  Prints one JSON
document (and writes it to --out)."""
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

from phyloligo_b200 import _lib, engine, phyloselect, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def progress(msg):
    print(msg, file=sys.stderr, flush=True)


def fit(D, method):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Z = phyloselect.linkage(D, method)
    torch.cuda.synchronize()
    return Z, time.perf_counter() - t0


def run(D, method, barrier_us):
    n = int(D.shape[0])
    out = {"method": method}
    progress("device %s, n = %d" % (method, n))
    torch.cuda.synchronize()
    _lib.timing_enable(True)
    _lib.timing_reset()
    t0 = time.perf_counter()
    _, _, _, phases = phyloselect.linkage_raw(D, method)  # synchronises on its status
    raw_s = time.perf_counter() - t0
    launch_ms, launches = _lib.timing_read(2)  # CUDA events around the cooperative launch alone
    _lib.timing_enable(False)
    assert launches == 1
    launch_s = launch_ms * 1e-3
    torch.cuda.empty_cache()
    Z, total_s = fit(D, method)
    torch.cuda.empty_cache()
    out.update({"fit_s": total_s, "linkage_raw_s": raw_s, "launch_s": launch_s, "phases": phases, "phases_per_n": phases / n,
                "us_per_phase": launch_s * 1e6 / phases, "barrier_floor_s": phases * barrier_us * 1e-6,
                "launch_over_floor": launch_s / (phases * barrier_us * 1e-6), "top_height": float(Z[-1, 2])})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--length", type=int, default=20_000)
    ap.add_argument("--sample", type=int, default=20_000, help="rows of the scipy comparison (0: skip)")
    ap.add_argument("--methods", default=",".join(phyloselect.LINKAGE_METHODS))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = engine.require_cuda()
    methods = args.methods.split(",")
    barrier_us = _lib.microbench(4)
    doc = {"card": card(), "barrier_us": barrier_us,
           "barrier_note": "po_microbench kind 4: microseconds per grid.sync() of an empty cooperative kernel on the "
                           "linkage kernels' largest grid (one 512-thread CTA per SM)",
           "workload": "%d contigs x %d bp (synth.device_fasta, seed 2), k=4 both strands, JSD float32 matrix resident (%.1f GB); "
                       "working copy float64 (%.1f GB) for all methods but single"
                       % (args.n, args.length, args.n * args.n * 4 / 1e9, args.n * args.n * 8 / 1e9)}
    text, b, e, _ = synth.device_fasta(args.n, args.length, 2, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    del text
    D = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    torch.cuda.synchronize()
    doc["runs"] = [run(D, m, barrier_us) for m in methods]
    if args.sample:
        m = min(args.sample, args.n)
        rows = np.sort(np.random.default_rng(0).choice(args.n, m, replace=False))
        idx = torch.from_numpy(rows).to(dev)
        S = D.index_select(0, idx).index_select(1, idx).contiguous()
        del D
        torch.cuda.empty_cache()
        from scipy.cluster.hierarchy import linkage as scipy_linkage
        from scipy.spatial.distance import squareform
        y = squareform(S.cpu().numpy(), checks=False)
        sample = {"rows": m, "how": "rows and columns of the matrix at %d seeded random indices (seed 0)" % m,
                  "cpu_threads": os.cpu_count(), "methods": []}
        for method in methods:
            progress("sample %s" % method)
            t0 = time.perf_counter()
            Zs = scipy_linkage(y, method)
            scipy_s = time.perf_counter() - t0
            fit(S, method)  # warm-up
            Zd, dev_s = fit(S, method)
            sample["methods"].append({"method": method, "scipy_cpu_s": scipy_s, "device_s": dev_s,
                                      "bitwise_equal": bool(np.array_equal(Zs, Zd, equal_nan=True))})
        doc["sample"] = sample
    out = json.dumps(doc, indent=1)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
