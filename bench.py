#!/usr/bin/env python3
"""Benchmark of the PhylOligo hot path on B200: profile a synthetic multi-FASTA and
compute its all-by-all JSD matrix (BASELINE.json: contig-pairs/sec, JSD k=4, strand both).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--scale S] [--dump-outputs DIR]

One "step" = one full pass over the workload: composition profiling of every
contig (k=4, both strands) + the JSD distance matrix.  Default workload is
BASELINE.json configs[1] (C2: 100 000 contigs x 20 kb); ``--scale`` shrinks the
contig count for quick checks (the JSON line then says so).  The input is drawn
from a fixed seed, so two builds run with the same arguments see the same bytes;
``--dump-outputs DIR`` writes what the last timed step computed (see dump_outputs)
so that their results can be compared.

`value`: unique contig pairs N(N+1)/2 resolved per second with the FASTA text
already resident in HBM and the matrix left in HBM.  `e2e`: the same pass from
pinned HOST memory (FASTA bytes -> host index -> H2D -> kernels -> every row
panel copied back D2H into pinned buffers), all inside the timed region.
Multi-GPU (torchrun): records are sharded for profiling, profiles all-gathered
over NCCL; the matrix is split in 2N block rows, rank s owns rows s and 2N-1-s
(equal rows, equal upper-triangle area), every rank computes only what lies
right of the diagonal and sends the transposed off-diagonal blocks to the
owners of those rows.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the benchmark leaves the source tree as it found it (it may be read-only): no bytecode caches
sys.dont_write_bytecode = True

METRIC = "contig-pairs/sec (JSD, k=4)"
UNIT = "pairs/s"
PATTERN = "1111"
STRAND = "both"
DIM = 256
JSD_FLOPS_PER_PAIR = 10 * DIM  # SURVEY.md 8(d) convention: 10 flop per dimension per pair
DUMP_RECORDS = 2048  # --dump-outputs: 2048 x 2048 float32 distances + 2048 x 256 float32 profiles, 18 MB


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the C2 contig count (1.0 = 100 000)")
    ap.add_argument("--mean-len", type=int, default=20_000)
    ap.add_argument("--panel-rows", type=int, default=4096)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.configs block (C3, C4, C5 kernels)")
    ap.add_argument("--no-cli", action="store_true", help="skip the e2e_cli leg (dispatcher functions into a real memmap file)")
    ap.add_argument("--ring-sink", action="store_true",
                    help="end to end: copy whole row panels into a 2-slot pinned ring instead of a host matrix")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the profiles and distances of the last one as DIR/<name>.npy "
                         "(one process only; a fixed sample of %d records when there are more)" % DUMP_RECORDS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    return args


def dump_outputs(out_dir, freq, matrix):
    """Write what a caller of the timed path receives, for comparing two builds output for output:
    profiles.npy  float32 (m, 256)  k=4 frequency profiles of the sampled records
    distances.npy float32 (m, m)    their JSD matrix (rows and columns of the sampled records)
    records.npy   float64 (m,)      which records: all of them when there are at most DUMP_RECORDS, else a
                                    seeded sample of DUMP_RECORDS - 2 plus the first and the last"""
    import torch

    n = int(matrix.shape[0])
    if n <= DUMP_RECORDS:
        idx = np.arange(n)
    else:
        idx = np.union1d(np.random.default_rng(0).choice(n, DUMP_RECORDS - 2, replace=False), [0, n - 1])
    d_idx = torch.from_numpy(idx).to(matrix.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"profiles": freq[d_idx].cpu().numpy(),
              "distances": matrix[d_idx[:, None], d_idx[None, :]].cpu().numpy(),
              "records": idx.astype(np.float64)}
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def workload_name(n, mean_len):
    return "C2: JSD k=4 strand=both, %d contigs x %d kb synthetic multi-FASTA" % (n, mean_len // 1000)


def workload_config(n, mean_len):
    """The `config` object of the JSON line: the same in both arms (ours and --impl reference)."""
    return {"workload": workload_name(n, mean_len), "pattern": PATTERN, "strand": STRAND, "contigs": n,
            "mean_contig_length": mean_len, "unique_pairs": n * (n + 1) // 2,
            "l2": "inputs (~%.2f GB of FASTA text) and outputs (%.1f GB matrix) exceed the 126 MB L2; no flush needed"
                  % (n * mean_len * 81 / 80 / 1e9, n * n * 4 / 1e9)}


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits", "-lms", "50",
                 "-i", str(self.gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                parts = [p.strip() for p in line.split(",")]
                if len(parts) < 9:
                    continue
                try:
                    sm.append(float(parts[1]))
                    smax.append(float(parts[2]))
                except ValueError:
                    continue
                for nm, val in zip(names, parts[5:9]):
                    if val.lower() == "active":
                        reasons.add(nm)
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(smax)), reasons=sorted(reasons), samples=len(sm))
        return out


# ---------------------------------------------------------------------------
# CPU baselines (the oracle port; the only place bench.py executes oracle/)
# ---------------------------------------------------------------------------
def _block_row_jsd(F, s):
    """One worker of the reference's block-row split: D(X[s], X) (distances_loc, bin/phyloligo.py:195-207)."""
    from sklearn.metrics import pairwise_distances
    from oracle import phylo_oracle as po
    return pairwise_distances(F[s], F, metric=po.JSD, n_jobs=1)


def cpu_python_port_rates(seqs_sample, n_profile, n_dist, n_jobs, modes=("serial",)):
    """Time the Python restatement of the reference path the way the reference runs it
    (joblib over sequences, bin/phyloligo.py:867-869; distances through sklearn.pairwise_distances
    with the callable metric, :388-390, or its block rows fanned out to joblib workers, :423-424).
    The distance stage is timed in every mode of `modes` and the FASTEST is kept, so that the
    baseline is not handicapped by the GIL: "serial" (one core; sklearn evaluates the upper
    triangle only), "threads" (pairwise_distances(n_jobs): threads in current sklearn) and
    "processes" (block rows over loky worker processes, what the reference's joblib did).
    Returns (seconds per base, seconds per unique pair, detail)."""
    from joblib import Parallel, delayed
    from sklearn.metrics import pairwise_distances
    from sklearn.utils import gen_even_slices
    from oracle import phylo_oracle as po

    prof = [s.decode("latin-1") for s in seqs_sample[:n_profile]]
    t0 = time.perf_counter()
    freqs = Parallel(n_jobs=n_jobs)(delayed(po.compute_frequency)(s, PATTERN, STRAND) for s in prof)
    t_prof = time.perf_counter() - t0
    bases = sum(len(s) for s in prof)
    F = np.vstack([np.asarray(f, dtype=np.float64) for f in freqs])
    if F.shape[0] < n_dist:  # cheap extra profiles for the distance sample
        extra = [po.frequency_np(s, PATTERN, STRAND) for s in seqs_sample[F.shape[0]:n_dist]]
        F = np.vstack([F] + extra) if extra else F
    F = F[:n_dist]
    n = F.shape[0]
    unique = n * (n + 1) // 2
    times = {}
    for mode in modes:
        t0 = time.perf_counter()
        if mode == "serial":
            D = pairwise_distances(F, metric=po.JSD, n_jobs=1)
        elif mode == "threads":
            D = pairwise_distances(F, metric=po.JSD, n_jobs=n_jobs)
        else:
            blocks = Parallel(n_jobs=n_jobs)(delayed(_block_row_jsd)(F, s) for s in gen_even_slices(n, n_jobs))
            D = np.vstack(blocks)
        times[mode] = time.perf_counter() - t0
        assert D.shape == (n, n)
    best = min(times, key=times.get)
    t_dist = times[best]
    return t_prof / max(1, bases), t_dist / max(1, unique), dict(
        profile_contigs=len(prof), profile_bases=bases, profile_s=t_prof, dist_rows=n, dist_s=t_dist,
        dist_mode=best, dist_seconds_by_mode=times)


def cpu_c_port_rates(seqs_sample, n_profile, n_dist, threads):
    """The same sample through the multi-threaded C restatement (oracle/oracle.c)."""
    from oracle import coracle
    from phyloligo_b200 import engine

    text, begin, end = engine.sequences_to_text(seqs_sample[:n_profile])
    t0 = time.perf_counter()
    F = coracle.profile_batch(text, begin, end, PATTERN, STRAND, threads=threads)
    t_prof = time.perf_counter() - t0
    bases = int((end - begin).sum())
    F = F[:n_dist]
    t0 = time.perf_counter()
    coracle.pairwise_rows("JSD", F, threads=threads)
    t_dist = time.perf_counter() - t0
    n = F.shape[0]
    return t_prof / max(1, bases), t_dist / max(1, n * n), dict(profile_bases=bases, profile_s=t_prof, dist_rows=n, dist_s=t_dist)


def ncu_traffic(n_contigs):
    """DRAM bytes per launch of the JSD tile kernel from the committed ncu --set full captures
    (profiles/r02_traffic.json), when one was taken at this problem size; else None."""
    try:
        recs = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))["jsd_tile_kernel"]
        for rec in recs if isinstance(recs, list) else [recs]:
            if rec["n_contigs"] == n_contigs:
                return rec["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def whole_job_pairs_per_s(n_contigs, total_bases, s_per_base, s_per_pair):
    pairs = n_contigs * (n_contigs + 1) // 2
    return pairs / (s_per_base * total_bases + s_per_pair * pairs)


def sample_sequences(n, mean_len, seed=2):
    from phyloligo_b200 import synth
    return synth.make_sequences(n, mean_len, seed=seed)


def run_reference(args):
    """--impl reference: the reference's CPU path (Python port of the joblib back-end,
    all host cores) on a bounded sample of the same workload; the value is the
    whole-job throughput those measured rates imply for the named workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_contigs = max(64, int(round(100_000 * args.scale)))
    total_bases = n_contigs * args.mean_len
    cores = os.cpu_count() or 1
    n_profile = min(n_contigs, max(64, 8 * cores))  # a few seconds of work per step on all cores
    n_dist = min(n_contigs, 600)
    seqs = sample_sequences(max(n_profile, n_dist), args.mean_len)
    vals, detail = [], None
    for it in range(args.warmup + args.steps):
        spb, spp, detail = cpu_python_port_rates(seqs, n_profile, n_dist, cores, modes=("serial", "threads", "processes"))
        if it >= args.warmup:
            vals.append((spb, spp))
    spb = float(np.mean([v[0] for v in vals]))
    spp = float(np.mean([v[1] for v in vals]))
    value = whole_job_pairs_per_s(n_contigs, total_bases, spb, spp)
    step_ms = 1e3 * (detail["profile_s"] + detail["dist_s"])
    sample = ("Python port of the reference joblib path on %d cores: %d contigs profiled by joblib worker processes, %d profiles "
              "all-pairs JSD timed three ways (serial / sklearn threads / block rows over joblib worker processes), fastest kept: "
              "%s (%s); value = whole-job pairs/s those rates imply for the workload"
              % (cores, n_profile, n_dist, detail["dist_mode"],
                 ", ".join("%s %.2f s" % kv for kv in sorted(detail["dist_seconds_by_mode"].items()))))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(n_contigs, args.mean_len),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "seconds_per_base": spb, "seconds_per_pair": spp},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def run_extra_configs(device, scale, hbm_peak, bf16_peak, fp32_peak):
    """BASELINE.json configs[2..4] on one GPU, device-resident kernels timed with CUDA events in this
    same process (same clocks record as the headline): C3 spaced pattern 111010011 (4096 dims) Eucl
    (Gram form, tensor cores) and BC on 50 000 reads x 15 kb; C4 Kendall / Spearman on 20 000
    tie-heavy short sequences; C5 JSD k=5 at N = 1 000 000 contigs x 5 kb on a stated sample of row
    panels (the 4 TB matrix is streamed panel by panel, never resident), extrapolated explicitly."""
    import torch
    from phyloligo_b200 import _lib, engine, synth
    from phyloligo_b200._lib import FLAG_MIRROR, FLAG_SKIP_LOWER

    def timed(fn, reps):
        fn()  # warm-up (first launch of a kernel configures its shared-memory opt-in)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def matrix_stage(X, metric, reps, flop_per_pair, peak, peak_unit, bound):
        n = int(X.shape[0])
        P, aux, dim = engine.prepare(X, metric)
        out = torch.empty((n, n), dtype=torch.float32, device=device)
        ms_prep = timed(lambda: engine.prepare(X, metric), 1)
        ms = timed(lambda: engine.distance_block(metric, P, aux, dim, 0, n, 0, n, out, 0, 0, FLAG_SKIP_LOWER | FLAG_MIRROR), reps)
        pairs = n * (n + 1) // 2
        tile = {"JSD": (32, 64), "EuclGram": (128, 128)}.get(metric, (64, 64))
        if metric == "SC" and 64 <= dim <= 4096:
            tile = (128, 128)
        computed = sum((min(n, t0 + tile[0]) - t0) * (n - (t0 // tile[1]) * tile[1]) for t0 in range(0, n, tile[0]))
        achieved = computed * flop_per_pair / (ms * 1e-3) / 1e12
        res = {"metric": metric, "kernel_ms": ms, "prepare_ms": ms_prep, "unique_pairs_per_s": pairs / (ms * 1e-3),
               "pairs_computed": computed,
               "roofline": {"bound": bound, "achieved": achieved, "peak": peak, "unit": peak_unit,
                            "frac": achieved / peak if peak else None, "work_per_pair": flop_per_pair}}
        del out, P, aux
        torch.cuda.empty_cache()
        return res

    extras = {}
    popc_peak = _lib.microbench(2)
    # ---- C3 ----
    n3 = max(256, int(round(50_000 * scale)))
    text, b, e, bases = synth.device_fasta(n3, 15_000, 3, device)
    prof = lambda: engine.profile_device(text, b, e, "111010011", "both", want=("freq32",))  # noqa: E731
    ms_prof = timed(prof, 2)
    X = prof()["freq32"]
    c3 = {"workload": "C3: pattern 111010011 (4096 dims) strand both, %d reads x 15 kb (fixed-length synthetic, generated on the device)" % n3,
          "profiling": {"kernel_ms": ms_prof, "gbases_per_s": bases / (ms_prof * 1e-3) / 1e9,
                        "roofline": {"bound": "hbm", "achieved": (int(text.shape[0]) + n3 * 4096 * 4) / (ms_prof * 1e-3) / 1e9,
                                     "peak": hbm_peak, "unit": "GB/s",
                                     "frac": (int(text.shape[0]) + n3 * 4096 * 4) / (ms_prof * 1e-3) / 1e9 / hbm_peak}},
          "stages": []}
    del text
    c3["stages"].append(matrix_stage(X, "EuclGram", 3, 2 * 4096, bf16_peak, "TFLOP/s", "tensor"))
    c3["stages"].append(matrix_stage(X, "BC", 1, 5 * 4096, fp32_peak, "TFLOP/s", "fp32"))
    extras["C3"] = c3
    del X
    torch.cuda.empty_cache()
    # ---- C4 ----
    n4 = max(256, int(round(20_000 * scale)))
    seqs = synth.make_sequences(n4, 375, 4, "short", all_n_frac=0.005)
    res = engine.profile_text(np.frombuffer(synth.to_fasta_bytes(seqs), dtype=np.uint8), "1111", "both", want=("freq32",))
    X = res["freq32"]
    c4 = {"workload": "C4: k=4 on %d tie-heavy short sequences (150-600 bp, 0.5 %% empty / all-N)" % n4, "stages": []}
    kt = matrix_stage(X, "KT", 2, 256 * 255 // 2, popc_peak * 16.0, "1e12 element-pair classifications/s", "popc")
    kt["roofline"]["note"] = ("work = D(D-1)/2 element-pair classifications per pair (SURVEY.md 8d); peak = measured POPC rate x 16 "
                              "(a 32-bit word classifies 32 element pairs with 2 POPC)")
    c4["stages"].append(kt)
    c4["stages"].append(matrix_stage(X, "SC", 3, 2 * 256, bf16_peak, "TFLOP/s", "tensor"))
    extras["C4"] = c4
    del X
    torch.cuda.empty_cache()
    # ---- C5 at N = 1M: a sample of row panels ----
    n5 = max(2048, int(round(1_000_000 * scale)))
    text, b, e, bases = synth.device_fasta(n5, 5_000, 5, device)
    prof = lambda: engine.profile_device(text, b, e, "11111", "both", want=("freq32",))  # noqa: E731
    ms_prof = timed(prof, 1)
    X = prof()["freq32"]
    text_bytes = int(text.shape[0])
    del text
    torch.cuda.empty_cache()
    P, aux, dim = engine.prepare(X, "JSD")
    rows = 1024
    bufs = [torch.empty((rows, n5), dtype=torch.float32, device=device) for _ in range(2)]
    ring = [torch.empty((rows, n5), dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    starts = [0, (n5 // 2) // rows * rows, max(0, (n5 - 4 * rows) // rows * rows)]
    kernel_ms, stream_ms = [], []
    for r_first in starts:
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        engine.distance_block("JSD", P, aux, dim, r_first, min(n5, r_first + rows), 0, n5, bufs[0], r_first, 0, 0)  # warm-up
        torch.cuda.synchronize()
        k0.record()
        engine.distance_block("JSD", P, aux, dim, r_first, min(n5, r_first + rows), 0, n5, bufs[0], r_first, 0, 0)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms.append(k0.elapsed_time(k1))
        # four consecutive panels, each copied to pinned host memory while the next one computes
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        free = [None, None]
        s0.record()
        for k in range(4):
            r0 = r_first + k * rows
            if r0 >= n5:
                break
            slot = k & 1
            if free[slot] is not None:
                torch.cuda.current_stream().wait_event(free[slot])
            engine.distance_block("JSD", P, aux, dim, r0, min(n5, r0 + rows), 0, n5, bufs[slot], r0, 0, 0)
            ready = torch.cuda.Event()
            ready.record()
            copy_stream.wait_event(ready)
            with torch.cuda.stream(copy_stream):
                ring[slot].copy_(bufs[slot], non_blocking=True)
                free[slot] = torch.cuda.Event()
                free[slot].record(copy_stream)
        torch.cuda.current_stream().wait_stream(copy_stream)
        s1.record()
        torch.cuda.synchronize()
        stream_ms.append(s0.elapsed_time(s1) / 4)
    km, sm_ = float(np.mean(kernel_ms)), float(np.mean(stream_ms))
    panels = -(-n5 // rows)
    achieved = rows * n5 * 10 * dim / (km * 1e-3) / 1e12
    extras["C5"] = {
        "workload": "C5: JSD k=5 (1024 dims) strand both, %d contigs x 5 kb (fixed-length synthetic, generated on the device), "
                    "--large memmap style row panels" % n5,
        "profiling": {"kernel_ms": ms_prof, "gbases_per_s": bases / (ms_prof * 1e-3) / 1e9,
                      "roofline": {"bound": "hbm", "achieved": (text_bytes + n5 * 1024 * 4) / (ms_prof * 1e-3) / 1e9, "peak": hbm_peak,
                                   "unit": "GB/s", "frac": (text_bytes + n5 * 1024 * 4) / (ms_prof * 1e-3) / 1e9 / hbm_peak}},
        "sample": "row panels of %d rows x %d columns at rows %s (every entry of the panel computed: the %.1f TB matrix is never "
                  "resident, so the symmetry shortcut does not apply); kernel alone, and 4 consecutive panels with the D2H of each "
                  "(%.1f GB into pinned memory) overlapped with the next" % (rows, n5, starts, n5 * n5 * 4 / 1e12, rows * n5 * 4 / 1e9),
        "kernel_ms_per_panel": kernel_ms, "streamed_ms_per_panel": stream_ms,
        "entries_per_s_kernel": rows * n5 / (km * 1e-3), "entries_per_s_streamed": rows * n5 / (sm_ * 1e-3),
        "extrapolation": {"panels": panels, "one_gpu_s": panels * sm_ * 1e-3, "eight_gpus_s": panels * sm_ * 1e-3 / 8,
                          "how": "panels x streamed ms per panel; row panels are independent, so 8 GPUs take 1/8 "
                                 "(host side: 4 TB through 8 x PCIe into the memmap)"},
        "roofline": {"bound": "fp32", "kernel": "jsd_tile_kernel<float>", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": achieved / fp32_peak if fp32_peak else None, "flop_convention": "10 flop per dimension per entry, D=1024"},
    }
    return extras


def run_select_leg(matrix, hbm_peak):
    """phyloselect's front half on the matrix that is resident after a step (SURVEY.md 8f rank 4): the
    K-medoids loop of bin/phyloselect.py:119-240 and the neighbour graph of its TSNE / HDBSCAN consumers
    (:381-428; default perplexity 100 -> 301 neighbours), all single passes over the N x N matrix in HBM."""
    import torch
    from phyloligo_b200 import phyloselect

    n = int(matrix.shape[0])
    nbytes = n * n * 4

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps, out

    ms_sum, _ = timed(lambda: phyloselect.row_sums(matrix))
    t0 = time.perf_counter()
    km = phyloselect.KMedoids(n_clusters=2).fit(matrix)
    torch.cuda.synchronize()
    fit_s = time.perf_counter() - t0
    k = min(301, n - 1)
    ms_knn, _ = timed(lambda: phyloselect.knn_graph(matrix, k), reps=1)
    return {
        "matrix": "%d x %d float32, resident after the distance stage" % (n, n),
        "row_sums_ms": ms_sum,
        "row_sums_roofline": {"bound": "hbm", "achieved": nbytes / (ms_sum * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                              "frac": nbytes / (ms_sum * 1e-3) / 1e9 / hbm_peak},
        "kmedoids": {"n_clusters": 2, "iterations": int(km.n_iter_), "seconds": fit_s,
                     "cluster_sizes": np.bincount(km.labels_, minlength=2).tolist(),
                     "passes_over_the_matrix": 1 + int(km.n_iter_), "note": "heuristic initialisation + one masked pass per iteration"},
        "knn": {"k": k, "ms": ms_knn, "gbytes_per_s_one_pass_equivalent": nbytes / (ms_knn * 1e-3) / 1e9,
                "note": "one pass over every row: threshold from an 8192-entry sample of the row, candidates below it sorted in "
                        "shared memory; the exact radix select (four histogram passes + a gather) is the fallback"},
    }


def run_cli_leg(fasta, n_contigs, pairs_unique, rank, world, device, want_rows):
    """The call a user of the reference makes: phyloligo.compute_frequencies(...) then
    phyloligo.compute_distances("joblib", "memmap", ...) (reference bin/phyloligo.py:980-997, 536-553)
    from a FASTA FILE into a raw float32 N x N FILE, wall clock, everything included (file read,
    host index, H2D, kernels, D2H, the host writing the file's pages).  Run twice: into a fresh file
    (the kernel has to instantiate every page of it) and again over the existing file."""
    import shutil
    import torch
    import torch.distributed as dist
    from phyloligo_b200 import phyloligo

    shm = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
    tag = "%s_%d" % (os.environ.get("MASTER_PORT", "0"), n_contigs)
    work = os.path.join(shm, "phyloligo_bench_cli_" + tag)
    genome = os.path.join(work, "assembly.fasta")
    out = os.path.join(work, "distances.mat")
    need = n_contigs * n_contigs * 4 + len(fasta) + (1 << 30)
    ok = 1
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)
        os.makedirs(work)
        if shutil.disk_usage(shm).free < need:
            ok = 0
        else:
            np.asarray(fasta).tofile(genome)
    if world > 1:
        flag = torch.tensor([ok], device=device)
        dist.broadcast(flag, 0)
        ok = int(flag.item())
    if not ok:
        return {"unavailable": "not enough room under %s for the %.1f GB output file" % (shm, need / 1e9)}
    cores = os.cpu_count() or 1
    runs = []
    for label in ("fresh file", "existing file"):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        freqs, fname = phyloligo.compute_frequencies("joblib", "memmap", genome, PATTERN, STRAND, 250, cores, work)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        phyloligo.compute_distances("joblib", "memmap", freqs, fname, out, "JSD", cores, 250, work)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t2 = time.perf_counter()
        runs.append({"output": label, "frequencies_s": t1 - t0, "distances_s": t2 - t1,
                     "pairs_per_s": pairs_unique / (t2 - t0)})
        del freqs
    res = None
    if rank == 0:
        m = np.memmap(out, dtype=np.float32, mode="r", shape=(n_contigs, n_contigs))
        for r, want in want_rows.items():
            assert np.array_equal(np.asarray(m[r]), want), "CLI leg: row %d of the file differs from the device result" % r
        assert not np.asarray(m[n_contigs // 2, n_contigs // 2 - 8:n_contigs // 2 + 8][8:9]).any()
        del m
        res = {"value": runs[0]["pairs_per_s"], "unit": UNIT, "runs": runs,
               "call": "phyloligo.compute_frequencies('joblib','memmap',...) + compute_distances('joblib','memmap',...): "
                       "FASTA file -> raw float32 N x N file under %s, wall clock" % shm,
               "output_bytes": n_contigs * n_contigs * 4,
               "note": "a fresh output file is bound by the kernel instantiating its pages (8-14 GB/s on this pool, "
                       "profiles/r02_sink_probe.log), not by PCIe (52 GB/s) or the kernels"}
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(work, ignore_errors=True)
    return res



def run_ours(args):
    # Libraries (NCCL's version banner, for one) write to stdout; the contract is ONE JSON line there.
    # Everything but that line goes to stderr: fd 1 points at stderr until the result is printed.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    import torch
    import torch.distributed as dist
    from phyloligo_b200 import _lib, engine, synth
    from phyloligo_b200._lib import FLAG_MIRROR, FLAG_SKIP_LOWER

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs needs a single process: under torchrun every rank holds only its rows of the matrix")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout (one JSON line only)
        dist.init_process_group("nccl", device_id=device)
        engine.bind_host_to_gpu_node(local_rank)  # pinned buffers in the memory next to this GPU (no-op on one node)
    _lib.load()

    n_contigs = max(64, int(round(100_000 * args.scale)))
    # synthetic input: generated once per node (rank 0) and shared through /dev/shm, so that N ranks
    # do not hold N copies of a multi-GB generator in host memory
    if world == 1:
        fasta, total_bases = synth.fast_fasta_bytes(n_contigs, args.mean_len, seed=2)
    else:
        shm_dir = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
        shm_path = os.path.join(shm_dir, "phyloligo_bench_%s_%d_%d.npy" % (os.environ.get("MASTER_PORT", "0"), n_contigs, args.mean_len))
        meta = torch.zeros(1, dtype=torch.int64, device=device)
        if rank == 0:
            fasta0, total_bases = synth.fast_fasta_bytes(n_contigs, args.mean_len, seed=2)
            np.save(shm_path, fasta0)
            del fasta0
            meta[0] = total_bases
        dist.broadcast(meta, 0)  # also the barrier that makes the file visible
        total_bases = int(meta.item())
        fasta = np.load(shm_path, mmap_mode="r")
    pairs_unique = n_contigs * (n_contigs + 1) // 2

    # ---- sharding: contiguous record ranges balanced by bytes; triangle-balanced block rows ----
    from phyloligo_b200 import multigpu, sharding
    begin_all, end_all = engine.fasta_index(fasta)
    assert begin_all.shape[0] == n_contigs
    cuts = sharding.record_cuts(end_all - begin_all, world)
    rec_lo, rec_hi = cuts[rank], cuts[rank + 1]
    n_local = rec_hi - rec_lo
    n_max = max(cuts[r + 1] - cuts[r] for r in range(world))
    # a shard starts at the '>' of its first record (= where the previous record's range ends)
    byte_lo = (int(end_all[rec_lo - 1]) if rec_lo > 0 else 0) if n_local else 0
    byte_hi = int(end_all[rec_hi - 1]) if n_local else 0
    pinned_text = torch.from_numpy(fasta[byte_lo:byte_hi].copy()).pin_memory()
    shard_bytes = byte_hi - byte_lo
    panel = max(64, (args.panel_rows // 64) * 64)
    symmetric = world == 1
    # block rows: rank s owns ranges s and 2*world-1-s (equal rows and equal upper-triangle area)
    ranges = sharding.paired_row_ranges(n_contigs, world)
    rows_owned = sum(ranges[i][1] - ranges[i][0] for i in sharding.owned_ranges(ranges, rank, world))

    # persistent device buffers
    d_text = torch.empty(shard_bytes + 64, dtype=torch.uint8, device=device)
    d_text[shard_bytes:].fill_(10)
    d_text[:shard_bytes].copy_(pinned_text)
    d_begin = torch.from_numpy(begin_all[rec_lo:rec_hi] - byte_lo).to(device)
    d_end = torch.from_numpy(end_all[rec_lo:rec_hi] - byte_lo).to(device)
    freq_pad = torch.zeros((n_max, DIM), dtype=torch.float32, device=device)
    gathered = torch.empty((world * n_max, DIM), dtype=torch.float32, device=device) if world > 1 else None
    if symmetric:
        matrix = torch.empty((n_contigs, n_contigs), dtype=torch.float32, device=device)
        job = None
    else:
        # this rank's rows; the other ranks' transposed tiles land in them over NVLink (peer memory)
        job = multigpu.BlockRows(n_contigs, torch.float32, rank, world)
        matrix = job.matrix
    # end-to-end sink: the result matrix (this rank's rows of it) in pinned host memory when the host has
    # room for it, else a 2-slot ring of row panels (discard sink)
    host_rows_n = n_contigs if symmetric else max(1, rows_owned)
    host_bytes = host_rows_n * n_contigs * 4
    try:
        avail = int([l for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0].split()[1]) * 1024
    except Exception:
        avail = 0
    host_result = None
    shared_host = None   # world > 1: (FileMatrix, n x n host tensor every rank maps, MirroredHostSink pool)
    if world > 1 and not args.ring_sink and not os.environ.get("PO_BENCH_RANK_ROWS") and n_contigs * n_contigs * 4 < 0.5 * avail:
        # One n x n matrix in shared memory that every rank maps; a rank page-locks its own rows (the DMA
        # target).  Only the parts of the block rows on and right of the diagonal cross PCIe; the rank that
        # shipped a block transposes it into the rows below (multigpu.MirroredHostSink).
        from phyloligo_b200 import hostsink
        shm_dir2 = "/dev/shm" if os.path.isdir("/dev/shm") else tempfile.gettempdir()
        e2e_path = os.path.join(shm_dir2, "phyloligo_bench_e2e_%s_%d.mat" % (os.environ.get("MASTER_PORT", "0"), n_contigs))
        ok = 1
        fm = None
        if rank == 0:
            try:
                fm = hostsink.FileMatrix(e2e_path, n_contigs, n_contigs, np.float32, create=True)
                os.posix_fallocate(fm.fd, 0, fm.nbytes)
            except Exception as exc:
                print("bench: no shared host matrix (%s)" % exc, file=sys.stderr)
                ok = 0
        dist.barrier()  # the file exists (or rank 0 has given up: the all-reduce below tells everybody)
        try:
            if rank != 0:
                fm = hostsink.FileMatrix(e2e_path, n_contigs, n_contigs, np.float32, create=False)
            own = [ranges[i] for i in sharding.owned_ranges(ranges, rank, world) if ranges[i][1] > ranges[i][0]]
            if ok and not fm.register_rows(own):
                print("bench: rank %d cannot page-lock its rows of the shared host matrix (%s)"
                      % (rank, _lib.load().po_last_error().decode(errors="replace")), file=sys.stderr)
                ok = 0
        except Exception as exc:
            print("bench: rank %d: no shared host matrix (%s)" % (rank, exc), file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 1:
            threads = int(os.environ.get("PO_HOST_MIRROR_THREADS", "0")) or max(2, -(-3 * (os.cpu_count() or 1) // (2 * world)))
            host_all = torch.from_numpy(fm.array)
            pool_ = engine.HostMirror(threads)
            shared_host = (fm, host_all, pool_, multigpu.MirroredHostSink(host_all, pool_))
        else:
            if fm is not None:
                fm.close()
            fm = None
        dist.barrier()
        if rank == 0 and shared_host is None:
            try:
                os.unlink(e2e_path)
            except OSError:
                pass
    if shared_host is None and not args.ring_sink and host_bytes * world < 0.5 * avail:
        try:
            host_result = torch.empty((host_rows_n, n_contigs), dtype=torch.float32).pin_memory()
        except RuntimeError as exc:  # page-locking refused (cgroup / ulimit): fall back to the panel ring
            print("bench: cannot pin %.1f GB of host memory (%s); using the ring sink" % (host_bytes / 1e9, exc),
                  file=sys.stderr)
            host_result = None
    if world > 1 and shared_host is None:  # every rank must take the same path (the barriers inside BlockRows.compute are collective)
        flag = torch.tensor([1 if host_result is not None else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            host_result = None
    pin_ring = None
    if host_result is None and shared_host is None:
        pin_ring = [torch.empty((panel, n_contigs), dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    pin_begin = torch.from_numpy(np.zeros(max(1, n_local), dtype=np.int64)).pin_memory()
    pin_end = torch.from_numpy(np.zeros(max(1, n_local), dtype=np.int64)).pin_memory()

    def profile_and_gather(b, e):
        """profile this rank's records, return the full (n_contigs, DIM) float32 matrix"""
        if n_local:
            res = engine.profile_device(d_text, b, e, PATTERN, STRAND, want=("freq32",))
            freq_pad[:n_local].copy_(res["freq32"])
        if world == 1:
            return freq_pad[:n_contigs]
        dist.all_gather_into_tensor(gathered, freq_pad)
        parts = [gathered[r * n_max: r * n_max + (cuts[r + 1] - cuts[r])] for r in range(world)]
        return torch.cat(parts, dim=0)

    def d2h_panels(src_rows, n_rows):
        """copy finished rows to the pinned ring, panel by panel (discard sink)"""
        events = [None, None]
        d2h_bytes = 0
        for k, r0 in enumerate(range(0, n_rows, panel)):
            m = min(panel, n_rows - r0)
            slot = k & 1
            if events[slot] is not None:
                events[slot].synchronize()  # the host consumer is done with this slot
            pin_ring[slot][:m].copy_(src_rows[r0:r0 + m], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record()
            events[slot] = ev
            d2h_bytes += m * n_contigs * 4
        return d2h_bytes

    def distance_panels(X, d2h):
        """this rank's share of the matrix; with d2h every finished row panel goes to pinned host memory"""
        P, aux, dim = engine.prepare(X, "JSD")
        if symmetric and not d2h:
            engine.distance_block("JSD", P, aux, dim, 0, n_contigs, 0, n_contigs, matrix, 0, 0,
                                  FLAG_SKIP_LOWER | FLAG_MIRROR)
            return 0
        if symmetric and host_result is not None:
            # every panel's finished blocks (its rows right of the diagonal + the mirrored column block
            # below) leave for the host matrix while the next panel computes
            return engine.matrix_to_host(None, "JSD", host_result, torch.float32, panel, prepared=(P, aux, dim),
                                         device_matrix=matrix, stats=e2e_stats)
        if symmetric:
            # panel p is complete once computed (earlier panels mirrored its left part): copy it out
            # on the copy stream while panel p+1 computes
            d2h_bytes = 0
            events = [None, None]
            for k, r0 in enumerate(range(0, n_contigs, panel)):
                r1 = min(n_contigs, r0 + panel)
                m = r1 - r0
                engine.distance_block("JSD", P, aux, dim, r0, r1, 0, n_contigs, matrix, 0, 0,
                                      FLAG_SKIP_LOWER | FLAG_MIRROR)
                ready = torch.cuda.Event()
                ready.record()
                slot = k & 1
                if events[slot] is not None:
                    events[slot].synchronize()
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(ready)
                    pin_ring[slot][:m].copy_(matrix[r0:r1], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(copy_stream)
                    events[slot] = ev
                d2h_bytes += m * n_contigs * 4
            torch.cuda.current_stream().wait_stream(copy_stream)
            return d2h_bytes
        # multi-GPU: per owned block row the diagonal block (mirrored in place) and the blocks right of
        # it, whose transposed tiles the kernel stores into the owning rank's rows (multigpu.BlockRows)
        if d2h and shared_host is not None:
            sink = shared_host[3]
            sink.reset()
            job.compute("JSD", P, aux, dim, ship=sink.ship, left_parts=False, panel_rows=panel)
            sink.finish()
            e2e_stats.update(dma_bytes=sink.dma_bytes, host_mirrored_bytes=sink.mirrored_bytes,
                             mirror_threads=shared_host[2].threads)
            return sink.dma_bytes
        if d2h and host_result is not None:
            job.compute("JSD", P, aux, dim, host_rows=host_result, panel_rows=panel)
            return rows_owned * n_contigs * 4
        job.compute("JSD", P, aux, dim)
        return d2h_panels(matrix, rows_owned) if d2h else 0

    def step_resident():
        X = profile_and_gather(d_begin, d_end)
        distance_panels(X, d2h=False)

    e2e_bytes = {"h2d": 0, "d2h": 0}
    e2e_stats = {}  # engine.matrix_to_host: bytes over PCIe / bytes the host mirrored from what had arrived

    def step_e2e():
        # host: index this rank's FASTA bytes; H2D: text + index; kernels; D2H: every panel
        d_text[:shard_bytes].copy_(pinned_text, non_blocking=True)  # the text crosses PCIe while the host indexes it
        b, e = engine.fasta_index(pinned_text.numpy())
        pin_begin[:len(b)].copy_(torch.from_numpy(b))
        pin_end[:len(e)].copy_(torch.from_numpy(e))
        db = pin_begin[:len(b)].to(device, non_blocking=True)
        de = pin_end[:len(e)].to(device, non_blocking=True)
        X = profile_and_gather(db, de)
        d2h = distance_panels(X, d2h=True)
        e2e_bytes["h2d"] = shard_bytes + 16 * len(b)
        e2e_bytes["d2h"] = d2h

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def matrix_row(r):
        """row r of the distance matrix recomputed on this device (float32), for checking the file of the CLI leg"""
        X = profile_and_gather(d_begin, d_end)
        P, aux, dim = engine.prepare(X, "JSD")
        blk = torch.empty((1, n_contigs), dtype=torch.float32, device=device)
        engine.distance_block("JSD", P, aux, dim, r, r + 1, 0, n_contigs, blk, r, 0)
        return blk[0].cpu().numpy()

    def host_equals_device(host_rows, dev_rows, what):
        """every entry of the host result against the device result, bit for bit: the host rows go back to the
        device in chunks (outside the timed region)"""
        chunk = max(1, (256 << 20) // (n_contigs * 4))
        buf = torch.empty((chunk, n_contigs), dtype=torch.float32, device=device)
        for r0 in range(0, int(host_rows.shape[0]), chunk):
            r1 = min(int(host_rows.shape[0]), r0 + chunk)
            engine.copy2d(buf[:r1 - r0], host_rows[r0:r1])
            assert torch.equal(buf[:r1 - r0], dev_rows[r0:r1]), "%s differs from the device result in rows [%d, %d)" % (what, r0, r1)

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident measurement ----
    for _ in range(args.warmup):
        step_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    _lib.timing_reset()
    _lib.timing_enable(True)
    launches0 = _lib.launch_count()
    ms_total = timed(step_resident, args.steps)
    launches = _lib.launch_count() - launches0
    _lib.timing_enable(False)
    dist_ms, dist_n = _lib.timing_read(1)
    prof_ms, prof_n = _lib.timing_read(0)
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = ms_total / args.steps
    value = pairs_unique / (ms_per_step * 1e-3)
    if args.dump_outputs:  # the buffers still hold the last timed step's results
        dump_outputs(args.dump_outputs, freq_pad[:n_contigs], matrix)

    # ---- end to end (host buffers in, host buffers out) ----
    for _ in range(max(1, min(2, args.warmup))):
        step_e2e()
    # CUDA events bracket the whole region: the host-side indexing shows up as stream idle time
    e2e_s = torch.tensor([timed(step_e2e, args.steps) * 1e-3 / args.steps], dtype=torch.float64, device=device)
    e2e_value = pairs_unique / float(e2e_s.item())
    if host_result is not None:  # the host copy is the device result (spot check, outside the timed region)
        torch.cuda.synchronize()
        picks = sorted(set(int(v) for v in np.linspace(0, host_rows_n - 1, 41)))
        for r in picks:
            assert torch.equal(host_result[r], matrix[r].cpu()), "end-to-end host matrix differs from the device matrix in row %d" % r
        host_equals_device(host_result, matrix[:host_rows_n], "end-to-end host matrix")  # every entry, bit for bit
    if shared_host is not None:  # after timed()'s closing barrier every rank's share is in the shared matrix
        torch.cuda.synchronize()
        for i in job.my_ranges:
            a, b = job.ranges[i]
            for r in sorted(set(int(v) for v in np.linspace(a, b - 1, 9))):
                assert torch.equal(shared_host[1][r], job.out_rows[i][r - a].cpu()), \
                    "end-to-end shared host matrix differs from the device rows in row %d" % r
            host_equals_device(shared_host[1][a:b], job.out_rows[i], "shared host matrix, rows [%d, %d)" % (a, b))
    io_bytes = torch.tensor([e2e_bytes["h2d"], e2e_bytes["d2h"], e2e_stats.get("host_mirrored_bytes", 0)],
                            dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(io_bytes, op=dist.ReduceOp.SUM)

    select_leg = None
    if world == 1 and not args.no_extra:
        try:
            hbm_for_select = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
        except Exception:
            hbm_for_select = 6650.0
        step_resident()  # the matrix of a fresh step
        select_leg = run_select_leg(matrix, hbm_for_select)

    # ---- the drop-in path itself: compute_frequencies + compute_distances(... "memmap" ...) into a real file ----
    e2e_cli = None
    peer_exchange = job is not None and job.peers is not None
    had_host_result = host_result is not None or shared_host is not None
    had_shared_host = shared_host is not None
    if shared_host is not None:
        if world > 1:
            dist.barrier()  # nobody unmaps while another rank's pool may still write into these rows
        shared_host[2].close()
        fm_ = shared_host[0]
        shared_host = None
        fm_.close()
        if world > 1:
            dist.barrier()
        if rank == 0:
            try:
                os.unlink(e2e_path)
            except OSError:
                pass
    if not args.no_cli:
        sample_rows = [0, n_contigs // 3, n_contigs - 1]
        want_rows = {r: matrix_row(r) for r in sample_rows}  # collective under torchrun (all-gather of profiles)
        host_result = pin_ring = None
        matrix = None
        if job is not None:
            job.close()
            job = None
        torch.cuda.empty_cache()
        e2e_cli = run_cli_leg(fasta, n_contigs, pairs_unique, rank, world, device, want_rows)

    if rank == 0:
        # roofline of the dominant kernel (JSD tile kernel): algorithmic flop per launch / launch time
        pairs_per_step_computed = 0
        if symmetric:
            for t0_ in range(0, n_contigs, 64):
                pairs_per_step_computed += (min(n_contigs, t0_ + 64) - t0_) * (n_contigs - t0_)
        else:
            pairs_per_step_computed = sharding.upper_area(ranges, rank, world, n_contigs)
        launches_per_step = max(1, dist_n // max(1, args.steps))
        avg_launch_ms = dist_ms / max(1, dist_n)
        flop_per_launch = JSD_FLOPS_PER_PAIR * pairs_per_step_computed / launches_per_step
        achieved = flop_per_launch / (avg_launch_ms * 1e-3) / 1e12 if avg_launch_ms > 0 else 0.0
        fp32_peak = _lib.microbench(0)
        mufu_peak = _lib.microbench(1)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        prof_bytes = shard_bytes + n_local * DIM * 4
        prof_gbs = prof_bytes / (prof_ms / max(1, prof_n) * 1e-3) / 1e9 if prof_ms > 0 else 0.0
        mirror_note = ""
        if had_shared_host:
            mirror_note = ("; ONE n x n matrix in shared memory mapped by every rank (own rows page-locked): only the parts of the "
                           "block rows on and right of the diagonal cross PCIe (%.1f GB over all ranks), the rank that shipped a "
                           "block transposes it into the rows below from host memory (%.1f GB, %d threads per rank, "
                           "po_host_mirror_*, released in stream order, inside the timed region)"
                           % (io_bytes[1].item() / 1e9, io_bytes[2].item() / 1e9, e2e_stats.get("mirror_threads", 0)))
        elif e2e_stats.get("host_mirrored_bytes"):
            mirror_note = ("; %.1f GB of the entries left of the diagonal (share %.2f of every panel's mirrored column block) are "
                           "not copied but transposed on the host from the blocks that have arrived, by %d threads "
                           "(po_host_mirror_*), released in stream order, inside the timed region"
                           % (e2e_stats["host_mirrored_bytes"] / 1e9, engine.default_host_mirror_share(), e2e_stats["mirror_threads"]))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n_contigs, args.mean_len),
            "detail": {
                "total_bases": total_bases,
                "pairs_computed_per_step_rank0": pairs_per_step_computed,
                "parallelism": "1 GPU, upper triangle + mirror" if world == 1 else
                               "%d ranks: records sharded, NCCL all-gather of profiles, paired block rows (s, 2W-1-s), "
                               "transposed off-diagonal tiles %s" % (world, "stored by the tile kernel into the owner's rows over NVLink "
                               "(CUDA IPC peer memory)" if peer_exchange else "exchanged over NCCL send/recv"),
                "e2e_sink": ("the result matrix in pinned host memory (%.1f GB%s); finished blocks leave by strided "
                             "DMA (po_copy2d_async) while the next panel computes%s"
                             % ((n_contigs * n_contigs * 4 if had_shared_host else host_bytes) / 1e9,
                                "" if had_shared_host else " per rank", mirror_note)) if had_host_result
                            else "row panels of %d rows copied D2H into a 2-slot pinned ring (discard sink)" % panel,
            },
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                       "samples": clocks["samples"]},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(io_bytes[0].item()),
                    "d2h_bytes_per_step": int(io_bytes[1].item()), "ms_per_step": float(e2e_s.item()) * 1e3,
                    # entries left of the diagonal that did not cross PCIe: host threads transposed them from the
                    # blocks that had arrived (po_host_mirror_*), inside the timed region
                    "host_mirrored_bytes_per_step": int(io_bytes[2].item()),
                    "host_mirror_threads": int(e2e_stats.get("mirror_threads", 0)),
                    "host_result_bytes": (n_contigs * n_contigs * 4 if had_shared_host else int(host_bytes) * world) if had_host_result else 0},
            "gpu_launches": int(launches),
            "roofline": {
                "kernel": "jsd_tile_kernel<float>", "bound": "fp32",
                "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                "frac": achieved / fp32_peak if fp32_peak else None, "traffic": ncu_traffic(n_contigs),
                "peak_source": "po_microbench FFMA peak measured in this run (MEASURED_PEAKS.json has no FP32-pipe figure)",
                "flop_convention": "10 flop per dimension per pair (SURVEY.md 8d); D=256",
                "avg_launch_ms": avg_launch_ms, "launches_timed": int(dist_n),
                "mufu_lg2_peak_Tops": mufu_peak,
                "recipe_note": "the kernel spends 10 (chunks whose value ranges prove u <= 1/4) to 12 FP32-pipe operations "
                               "+ 1 MUFU per (pair, dimension) on a cancellation-free series; at 100 % FP32-pipe utilisation "
                               "that is 0.50 / 0.42 of the 10-flop convention, 0.465 for this workload's mix of chunk variants "
                               "(ncu: sm__pipe_fma_cycles_active 80.0 %, profiles/r02b_jsd_tile_full_ncu_summary.txt; DESIGN.md 4.3)",
            },
            "e2e_cli": e2e_cli,
            "stages": {
                "profiling_ms_per_launch": prof_ms / max(1, prof_n),
                "profiling_gbases_per_s_rank0": (total_bases * (n_local / n_contigs)) / (prof_ms / max(1, prof_n) * 1e-3) / 1e9
                if prof_ms > 0 else None,
                "profiling_roofline": {"bound": "hbm", "achieved": prof_gbs, "peak": hbm_peak, "unit": "GB/s",
                                       "frac": prof_gbs / hbm_peak, "bytes": prof_bytes},
                "distance_ms_per_step": dist_ms / max(1, args.steps),
            },
        }
        if world == 1 and not args.no_extra:
            bf16_peak = float(peaks.get("bf16_tflops", 1665.5))
            line["extra"] = {"select": select_leg,
                             "configs": run_extra_configs(device, args.scale, hbm_peak, bf16_peak, fp32_peak),
                             "peaks": {"hbm_gbs": hbm_peak, "bf16_tflops_burst": bf16_peak, "fp32_ffma_tflops": fp32_peak,
                                       "source": "MEASURED_PEAKS.json (HBM, bf16 burst); po_microbench in this run (FP32, POPC)"}}
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            # about 10-15 s of single-core CPU work: 300 contigs profiled (~1 us per base), 700 profiles all-pairs
            seqs = sample_sequences(700, args.mean_len)
            spb, spp, d1 = cpu_python_port_rates(seqs, 300, 700, 1)
            cval = whole_job_pairs_per_s(n_contigs, total_bases, spb, spp)
            cspb, cspp, d2 = cpu_c_port_rates(seqs, 700, 700, cores)
            line["cpu_baseline"] = {
                "value": cval, "unit": UNIT, "cores": 1, "kind": "port",
                "sample": "Python port of the reference path on 1 core: %d contigs profiled (%.1f s), %d profiles "
                          "all-pairs JSD (%.1f s); value = whole-job pairs/s those rates imply for this workload"
                          % (d1["profile_contigs"], d1["profile_s"], d1["dist_rows"], d1["dist_s"]),
                "seconds_per_base": spb, "seconds_per_pair": spp,
                "c_port": {"value": whole_job_pairs_per_s(n_contigs, total_bases, cspb, cspp), "unit": UNIT,
                           "cores": cores, "note": "multi-threaded C restatement (oracle/oracle.c): 700 contigs profiled, 700 profiles all-pairs"},
            }
        emit(line)
    if world > 1:
        if job is not None:
            job.close()
        dist.barrier()
        if rank == 0:
            try:
                os.unlink(shm_path)
            except OSError:
                pass
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the results of this project's path (--impl ours)")
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
