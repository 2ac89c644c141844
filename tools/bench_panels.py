"""Time phyloselect's row-panel passes (DESIGN.md 4.12) with CUDA events on one GPU.

    python tools/bench_panels.py [--out results.json] [--big 300000] [--file-gb 16]

1. C2's shape (100 000 profiles of 256 dimensions, JSD k = 4): the resident distance stage, then each consumer on
   the resident matrix and on forced profile panels (the neighbour graph, the t-SNE affinities, K-medoids k = 2,
   HDBSCAN min_cluster_size 5).
2. `--big` profiles (default 300 000, past the device): one neighbour-graph pass over profile panels, its pairs/s
   against the tile kernel's resident rate of step 1.  C5 (1 000 000 x 5 kb, k = 5: 1024 dimensions) is
   extrapolated from timed panels of its own shape.
3. The file source: GB/s of one pass (kNN) over a memmap file of `--file-gb` GB written just before (so in the
   page cache), read in panels.
Profiles are seeded random compositions; the card's name, power limit, clocks and throttle reasons are recorded.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from phyloligo_b200 import engine, panels, phyloselect  # noqa: E402
from phyloligo_b200._lib import TILE  # noqa: E402


def smi():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active,temperature.gpu"
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    except OSError as exc:
        return "nvidia-smi unavailable: %s" % exc


def timed(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / 1e3, out


def profiles(n, dim, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = torch.rand((n, dim), generator=g, device="cuda", dtype=torch.float32) ** 2
    return (X / X.sum(dim=1, keepdim=True)).contiguous()


def dump(res, out):
    if out:
        os.makedirs(os.path.dirname(out) or ".", exist_ok=True)
        with open(out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps(res), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the results to this JSON file")
    ap.add_argument("--n", type=int, default=100000)
    ap.add_argument("--big", type=int, default=300000)
    ap.add_argument("--file-gb", type=float, default=16.0)
    args = ap.parse_args()
    res = {"gpu_before": smi()}
    n = args.n
    X = profiles(n, 256, 1)
    phyloselect.knn_graph(engine.distance_matrix_device(X[:4096], "JSD", torch.float32), 10)  # warm-up
    t, D = timed(lambda: engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True))
    t, D = timed(lambda: engine.distance_matrix_device(X, "JSD", torch.float32, symmetric=True))
    pairs_res = n * (n + 1) / 2
    res["c2_resident_distance_s"] = t
    res["jsd_resident_pairs_per_s"] = pairs_res / t
    src = panels.ProfileSource(X, "JSD", panel_rows=8192)
    res["c2_panel_rows"] = src.panel_rows
    t_pass, _ = timed(lambda: [None for _ in src.panels()])
    res["c2_panel_pass_s"] = t_pass
    res["c2_panel_pass_over_resident_distance"] = t_pass / t
    res["c2_panel_pairs_per_s"] = n * n / t_pass
    rs = panels.ResidentSource(D)
    fits = {
        "knn_graph": lambda s: phyloselect.knn_graph(s, 10),
        "tsne_affinities": lambda s: phyloselect.tsne_affinities(s, 30.0),
        "kmedoids_k2": lambda s: phyloselect.KMedoids(n_clusters=2).fit(s).n_iter_,
        "hdbscan_mcs5": lambda s: int(phyloselect.HDBSCAN(min_cluster_size=5).fit(s).labels_.max()),
    }
    for name, fn in fits.items():
        tr, a = timed(lambda: fn(rs))
        tp, b = timed(lambda: fn(src))
        same = all(torch.equal(x, y) for x, y in zip(a, b)) if isinstance(a, tuple) else a == b
        res["c2_" + name] = {"resident_s": tr, "panels_s": tp, "same_result": bool(same)}
        print(name, res["c2_" + name], flush=True)
    del D, rs, src
    torch.cuda.empty_cache()
    dump(res, args.out)

    # past the device
    nb = args.big
    Xb = profiles(nb, 256, 2)
    big = panels.profile_source(Xb, "JSD")
    res["big_n"] = nb
    res["big_resident"] = big.resident
    res["big_panel_rows"] = big.panel_rows
    t, _ = timed(lambda: phyloselect.knn_graph(big, 10))
    res["big_knn_pass_s"] = t
    res["big_knn_pairs_per_s"] = nb * nb / t
    res["big_knn_rate_over_resident_tile_rate"] = (nb * nb / t) / res["jsd_resident_pairs_per_s"]
    dump(res, args.out)
    del big, Xb
    torch.cuda.empty_cache()

    # C5's shape: panels of 1 000 000 x 1024-dimension JSD profiles, timed on the first panels and extrapolated
    n5 = 1000000
    X5 = profiles(n5, 1024, 5)
    s5 = panels.ProfileSource(X5, "JSD", panel_rows=8192)
    it = s5.panels()
    next(it)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    k = 0
    for r0, r1, P in it:
        phyloselect._knn_rows(P, r0, 10, torch.empty((r1 - r0, 10), dtype=torch.int32, device="cuda"),
                              torch.empty((r1 - r0, 10), dtype=torch.float32, device="cuda"))
        k += 1
        if k == 4:
            break
    torch.cuda.synchronize()
    t = (time.perf_counter() - t0) / k
    res["c5_panel_rows"] = s5.panel_rows
    res["c5_timed_panels"] = k
    res["c5_s_per_panel"] = t
    res["c5_knn_pass_s_extrapolated"] = t * n5 / s5.panel_rows
    del s5, X5, it
    torch.cuda.empty_cache()
    dump(res, args.out)

    # the file source
    nf = int(np.sqrt(args.file_gb * 1e9 / 4)) // TILE * TILE
    Xf = profiles(nf, 256, 3)
    path = os.path.join(tempfile.mkdtemp(), "m.memmap")
    pf = panels.ProfileSource(Xf, "JSD")
    with open(path, "wb") as fh:
        for r0, r1, P in pf.panels():
            fh.write(P.cpu().numpy().tobytes())
    del pf
    torch.cuda.empty_cache()
    fsrc = panels.FileSource(path, nf)
    t, _ = timed(lambda: phyloselect.knn_graph(fsrc, 10))
    res["file_n"] = nf
    res["file_bytes"] = nf * nf * 4
    res["file_cached"] = "written just before the pass: in the page cache"
    res["file_panel_rows"] = fsrc.panel_rows
    res["file_knn_pass_s"] = t
    res["file_gb_per_s"] = nf * nf * 4 / t / 1e9
    fsrc.close()
    os.remove(path)
    res["gpu_after"] = smi()
    dump(res, args.out)


if __name__ == "__main__":
    main()
