#!/usr/bin/env python3
"""Time phyloselect's neighbour-joining trees (nj, bionj) on square samples of C2's resident JSD matrix (synthetic
contigs of 20 kb generated on the device, k=4 both strands, float32): for every size and method the whole fit
(input check, working state, every join, copy-back, as `fit_s`), the launches of po_nj_run from first to last (CUDA
events, timing family 3, `launches_s`), and the byte model of the two passes each join makes over the float64
working state: the row sums read 8 m^2 bytes, the Q scan 4 m^2 (about 12 m^2 per join, 4 n^3 per fit).  The
roofline share is that model over the measured time of the joins at m >= 20 000 (timed by running the fit on an
n-row sample and on a 20 000-row sample of it: the difference is the joins above 20 000 only approximately, since the
two samples differ; see `roofline_note`), against DESIGN.md's 6 650 GB/s HBM figure.  `us_per_join_small` is the
fit time per join at 2 000 rows, where the launches of a join, not bytes, set the pace.  For comparison the numpy
restatement (oracle/nj_oracle.py) on the CPU at 2 000 rows.  Prints one JSON document (and writes it to --out)."""
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

HBM_GBS = 6650.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def progress(msg):
    print(msg, file=sys.stderr, flush=True)


def model_bytes(n_from, n_to=3):
    """12 m^2 bytes per join for m = n_from down to n_to + 1."""
    m = np.arange(n_to + 1, n_from + 1, dtype=np.float64)
    return float((12.0 * m * m).sum())


def fit(D, method):
    torch.cuda.synchronize()
    _lib.timing_enable(True)
    _lib.timing_reset()
    t0 = time.perf_counter()
    edge, length, compactions = phyloselect.nj_raw(D, method)  # synchronises on its status
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms, launches = _lib.timing_read(3)
    _lib.timing_enable(False)
    assert launches == 1
    return edge, length, compactions, wall, ms * 1e-3


def sample(D, m, seed):
    rows = np.sort(np.random.default_rng(seed).choice(int(D.shape[0]), m, replace=False))
    idx = torch.from_numpy(rows).to(D.device)
    return D.index_select(0, idx).index_select(1, idx).contiguous()


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--n", type=int, default=50_000, help="contigs of the resident matrix")
    ap.add_argument("--length", type=int, default=20_000)
    ap.add_argument("--sizes", default="20000,50000")
    ap.add_argument("--methods", default="nj,bionj")
    ap.add_argument("--cpu-rows", type=int, default=2000, help="rows of the numpy restatement's CPU timing (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = engine.require_cuda()
    sizes = [int(s) for s in args.sizes.split(",") if s]
    methods = args.methods.split(",")
    doc = {"card": card(), "hbm_gbs": HBM_GBS,
           "workload": "square samples (seeded rows, seed 0) of the JSD float32 matrix of %d contigs x %d bp (synth.device_fasta, "
                       "seed 2), k=4 both strands" % (args.n, args.length),
           "model": "12 m^2 bytes per join (row sums 8 m^2, Q scan 4 m^2) over the float64 working state"}
    text, b, e, _ = synth.device_fasta(args.n, args.length, 2, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    del text
    D = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    torch.cuda.synchronize()
    small = sample(D, 2000, 1)
    for method in methods:  # warm-up
        fit(small, method)
    runs = []
    for method in methods:
        _, _, _, wall, launches_s = fit(small, method)
        runs.append({"rows": 2000, "method": method, "fit_s": wall, "launches_s": launches_s, "us_per_join_small": wall / 1997 * 1e6})
    for m in sizes:
        S = sample(D, m, 0) if m < args.n else D
        for method in methods:
            progress("%s at %d rows" % (method, m))
            edge, length, compactions, wall, launches_s = fit(S, method)
            torch.cuda.empty_cache()
            r = {"rows": m, "method": method, "fit_s": wall, "launches_s": launches_s, "compactions": compactions,
                 "model_bytes": model_bytes(m), "model_s_at_hbm": model_bytes(m) / (HBM_GBS * 1e9),
                 "model_over_launches": model_bytes(m) / (HBM_GBS * 1e9) / launches_s,
                 "root_lengths": length[-3:].cpu().numpy().tolist()}
            if m > 20000:
                sub = sample(S, 20000, 3)
                _, _, _, _, sub_s = fit(sub, method)
                del sub
                torch.cuda.empty_cache()
                big = model_bytes(m, 20000)
                r.update({"joins_above_20000_s": launches_s - sub_s, "joins_above_20000_bytes": big,
                          "joins_above_20000_gbs": big / (launches_s - sub_s) / 1e9,
                          "joins_above_20000_hbm_share": big / (launches_s - sub_s) / 1e9 / HBM_GBS})
            runs.append(r)
            progress(json.dumps(r))
        del S
        torch.cuda.empty_cache()
    doc["runs"] = runs
    doc["roofline_note"] = ("joins_above_20000: the fit at m rows minus the fit on a 20 000-row sample of it, against the "
                            "byte model of the joins m .. 20 001")
    if args.cpu_rows:
        from oracle import nj_oracle
        C = small.cpu().numpy() if args.cpu_rows == 2000 else sample(D, args.cpu_rows, 1).cpu().numpy()
        cpu = {"rows": args.cpu_rows, "what": "numpy restatement (oracle/nj_oracle.py) on the host, not ape", "cpu_threads": os.cpu_count()}
        for method in methods:
            t0 = time.perf_counter()
            want_e, want_l = nj_oracle.nj(C, method)
            cpu[method + "_s"] = time.perf_counter() - t0
            got_e, got_l = phyloselect.nj(torch.from_numpy(C).to(dev), method)
            cpu[method + "_device_bitwise_equal"] = bool(np.array_equal(want_e, got_e) and np.array_equal(want_l.view(np.uint64),
                                                                                                          got_l.view(np.uint64)))
        doc["cpu"] = cpu
    out = json.dumps(doc, indent=1)
    print(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(out + "\n")


if __name__ == "__main__":
    main()
