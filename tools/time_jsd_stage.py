#!/usr/bin/env python3
"""Time the C2 distance stage alone: the JSD matrix of bench.py's headline input (100 000 synthetic contigs
x 20 kb, seed 2, k=4 both strands, float32, symmetric: upper tiles computed, mirrored below), with CUDA events
around each po_distance_block launch.  The profiles and the prepared operands are made once, outside the timed
window; --reps full matrices are timed after one warm-up.  Also prints:
  - a fingerprint of the whole matrix (sum of its float32 bit patterns, and sha256 of its first 256 rows), so
    that two builds can be compared for bitwise equality without writing 40 GB;
  - the operand-bandwidth microbenchmarks (po_microbench kinds 5..12, and 0 and 3 for reference) with --microbench;
  - the card, its power limit and the SM clock and throttle reasons before and after.
Prints one JSON document (and writes it to --out)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from phyloligo_b200 import _lib, engine, synth  # noqa: E402
from phyloligo_b200._lib import FLAG_MIRROR, FLAG_SKIP_LOWER  # noqa: E402


def smi(fields):
    q = subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[:1]


def fingerprint(M, rows=4096):
    s = 0
    for r0 in range(0, M.shape[0], rows):
        s += int(M[r0:r0 + rows].view(torch.int32).to(torch.int64).sum().item())
    head = hashlib.sha256(M[:256].cpu().numpy().tobytes()).hexdigest()
    return {"bit_sum": s, "sha256_first_256_rows": head}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--contigs", type=int, default=100_000)
    ap.add_argument("--mean-len", type=int, default=20_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--microbench", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    torch.cuda.set_device(0)
    doc = {"card": {"torch_name": torch.cuda.get_device_name(0),
                    "nvidia_smi": smi("name,power.limit,clocks.max.sm")},
           "library": _lib.LIB_PATH}
    if args.microbench:
        names = {0: "FFMA TFLOP/s", 3: "MUFU.RCP 1e12 op/s",
                 5: "FFMA2 3 register pairs", 6: "FFMA2 2 register pairs + immediate",
                 7: "FFMA2 3 register pairs, shared operands (.reuse)", 8: "FFMA2 2 register pairs, shared multiplier (.reuse) + immediate",
                 9: "FFMA2 .F32 broadcast + immediate", 10: "FADD2 .F32 broadcast + register pair",
                 11: "FMUL2 x*x", 12: "V0 recipe, packed FP32 instructions"}
        doc["microbench"] = {"%d: %s" % (k, v): _lib.microbench(k) for k, v in names.items()}
        doc["microbench_units"] = "kinds 5..12: warp-instructions per SM per SM clock (clock measured in the kernel)"

    fasta, total_bases = synth.fast_fasta_bytes(args.contigs, args.mean_len, seed=2)
    X = engine.profile_text(fasta, "1111", "both", want=("freq32",))["freq32"]
    n = int(X.shape[0])
    P, aux, dim = engine.prepare(X, "JSD")
    M = torch.empty((n, n), dtype=torch.float32, device="cuda")

    def run():
        engine.distance_block("JSD", P, aux, dim, 0, n, 0, n, M, 0, 0, FLAG_SKIP_LOWER | FLAG_MIRROR)

    doc["clocks_before"] = smi("clocks.sm,clocks.max.sm,temperature.gpu,power.draw,clocks_throttle_reasons.active")
    run()
    torch.cuda.synchronize()
    ms = []
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run()
        e1.record()
        e1.synchronize()
        ms.append(e0.elapsed_time(e1))
    doc["clocks_after"] = smi("clocks.sm,clocks.max.sm,temperature.gpu,power.draw,clocks_throttle_reasons.active")
    pairs = n * (n + 1) // 2
    doc.update({"contigs": n, "dim": dim, "ms": ms, "ms_min": min(ms), "ms_median": float(np.median(ms)),
                "unique_pairs_per_s": pairs / (min(ms) * 1e-3), "fingerprint": fingerprint(M)})
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
