#!/usr/bin/env python3
"""Time phyloselect's t-SNE on the matrix resident after the distance stage, at C2's shape (100 000 contigs x 20 kb,
fixed-length synthetic FASTA generated on the device, k=4 both strands, JSD, float32), for perplexity 30 and 100:
the input check, the neighbour graph, the affinities (graph, perplexity search, symmetric CSR), the exact
repulsion pass per iteration (pairs/s against the bound of its binding pipe, with the FP32 and MUFU.RCP rates
measured by po_microbench in the same run), the attraction / step kernel and the whole 1000-iteration fit.  For
comparison, scikit-learn's TSNE on the CPU with its defaults (angle=0.5) on a 20 000-row sample of the same
matrix.  Prints one JSON document (and writes it to --out)."""
import argparse
import json
import os
import re
import shutil
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from phyloligo_b200 import _lib, engine, phyloselect, synth  # noqa: E402

# The repulsion kernel's inner loop (po_tsne.cu, unrolled 4 columns x 2 packed row pairs = 16 pairs per thread) is
# 32 FFMA2 + 24 FADD2 + 8 FMUL2 (= 128 FP32 lane operations), 16 MUFU.RCP and 4 LDS.128: per pair 8 FP32 lane
# operations and 1 MUFU.  The two-level float32 sums add 3 FADD2 per row pair per 32 columns (0.09 lane operations
# per pair), left out of the bound.
FP32_OPS_PER_PAIR = 8
MUFU_PER_PAIR = 1


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def sass_histogram():
    """Opcode counts of the repulsion kernel in the built library (whole function), if cuobjdump is at hand."""
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(tool):
        return None
    out = subprocess.run([tool, "-sass", _lib.LIB_PATH], capture_output=True, text=True).stdout
    m = re.search(r"Function : (\S*repulsion_kernel\S*)\n(.*?)(?:\n\s*\n\s*Function|\Z)", out, re.S)
    if not m:
        return None
    counts = {}
    for line in m.group(2).splitlines():
        op = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", line)
        if op:
            counts[op.group(1)] = counts.get(op.group(1), 0) + 1
    keep = ("FFMA2", "FADD2", "FMUL2", "MUFU", "LDS", "FFMA", "FADD", "FMUL")
    return {k: v for k, v in counts.items() if k in keep}


def event_ms(fn, reps=5):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run(D, perplexity, bound_pairs_s):
    n = int(D.shape[0])
    k = min(n - 1, int(3.0 * perplexity + 1))
    out = {"perplexity": perplexity, "k": k}
    out["check_ms"] = event_ms(lambda: phyloselect.check_tsne_matrix(D), reps=3)
    out["knn_ms"] = event_ms(lambda: phyloselect.knn_graph(D, k), reps=3)
    out["affinities_ms"] = event_ms(lambda: phyloselect.tsne_affinities(D, perplexity), reps=3)
    P = phyloselect.tsne_affinities(D, perplexity)
    out["nnz"] = int(P[2].numel())
    # repulsion and step at the positions of a short fit (a spread-out embedding, as in most iterations)
    t = phyloselect.TSNE(perplexity=perplexity, random_state=0, max_iter=300)
    Y0 = t.fit(D).embedding_
    st = phyloselect._Descent(P, Y0)
    lib = _lib.load()
    rep = lambda: lib.po_tsne_repulsion(phyloselect._ptr(st.Y), n, phyloselect._ptr(st.work), phyloselect._stream())  # noqa: E731
    out["repulsion_ms"] = event_ms(rep, reps=20)
    pairs_s = float(n) * n / (out["repulsion_ms"] * 1e-3)
    out["repulsion_pairs_per_s"] = pairs_s
    out["repulsion_frac_of_bound"] = pairs_s / bound_pairs_s
    step = lambda: st.gradient(12.0, 1.0, Y_next=st.Y_next, momentum=0.5, lr=2083.0)  # noqa: E731
    total = event_ms(lambda: step(), reps=20)
    out["attraction_step_ms"] = total - out["repulsion_ms"]
    out["attraction_step_note"] = "one repulsion + step call minus the repulsion pass alone"
    fit = phyloselect.TSNE(perplexity=perplexity, random_state=0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fit.fit(D)
    torch.cuda.synchronize()
    out["fit_s"] = time.perf_counter() - t0
    out["fit_n_iter"] = int(fit.n_iter_)
    out["fit_kl"] = float(fit.kl_divergence_)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__)
    ap.add_argument("--n", type=int, default=100_000)
    ap.add_argument("--length", type=int, default=20_000)
    ap.add_argument("--sample", type=int, default=20_000, help="rows of the scikit-learn comparison (0: skip)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    dev = engine.require_cuda()
    fp32_tflops = _lib.microbench(0)
    rcp_rate = _lib.microbench(3) * 1e12
    fp32_lane_ops = fp32_tflops * 1e12 / 2.0
    bounds = {"fp32_pairs_per_s": fp32_lane_ops / FP32_OPS_PER_PAIR, "mufu_pairs_per_s": rcp_rate / MUFU_PER_PAIR}
    bound = min(bounds.values())
    doc = {"card": card(), "microbench": {"ffma_tflops": fp32_tflops, "mufu_rcp_per_s": rcp_rate},
           "repulsion_per_pair": {"fp32_lane_ops": FP32_OPS_PER_PAIR, "mufu": MUFU_PER_PAIR}, "sass_repulsion_kernel": sass_histogram(),
           "bounds": bounds, "binding_pipe": min(bounds, key=bounds.get),
           "workload": "%d contigs x %d bp (synth.device_fasta, seed 2), k=4 both strands, JSD float32 matrix resident (%.1f GB)"
                       % (args.n, args.length, args.n * args.n * 4 / 1e9)}
    text, b, e, _ = synth.device_fasta(args.n, args.length, 2, dev)
    X = engine.profile_device(text, b, e, "1111", "both", want=("freq32",))["freq32"]
    del text
    D = engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True)
    torch.cuda.synchronize()
    doc["runs"] = [run(D, p, bound) for p in (30.0, 100.0)]
    if args.sample:
        m = min(args.sample, args.n)
        rows = np.sort(np.random.default_rng(0).choice(args.n, m, replace=False))
        idx = torch.from_numpy(rows).to(dev)
        S = D.index_select(0, idx).index_select(1, idx).contiguous()
        Sh = S.cpu().numpy().astype(np.float64)
        from sklearn.manifold import TSNE as SkTSNE
        t0 = time.perf_counter()
        sk = SkTSNE(metric="precomputed", init="random", random_state=0).fit(Sh)
        sk_s = time.perf_counter() - t0
        t = phyloselect.TSNE(random_state=0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        t.fit(S)
        torch.cuda.synchronize()
        dev_s = time.perf_counter() - t0
        doc["sample"] = {"rows": m, "how": "rows and columns of the matrix at %d seeded random indices (seed 0), float64 for "
                                           "scikit-learn" % m,
                         "sklearn_cpu_s": sk_s, "sklearn_kl": float(sk.kl_divergence_), "sklearn_angle": 0.5,
                         "device_s": dev_s, "device_kl": float(t.kl_divergence_), "cpu_threads": os.cpu_count()}
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
