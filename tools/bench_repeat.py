#!/usr/bin/env python
"""Repeat-detection kernel (SURVEY.md §8f #3, first half) on a window workload shaped like Lancet2's:
every window asked at each k of the graph's k-loop with two mismatches allowed, plus the exact check
at max_k.  Prints one JSON line: jobs/s through the C-ABI (host buffers, copies inside) and kernel-only,
k-mer-pair comparisons/s (the reference's unit of work), and the CPU arm (the reference's own
base/repeat.cpp from oracle/_ref when present, else the oracle port) on a bounded sample."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import repeat_lib  # noqa: E402
from lancet2_b200.repeat_scan import GpuRepeatScan  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=2000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--cpu-jobs", type=int, default=60)
    ap.add_argument("--library", default=None, help="a stand-alone build of lgr_repeat.cu instead of the main library (A/B runs)")
    args = ap.parse_args()
    kvals = tuple(range(13, 128, 6))          # Lancet2 defaults: min_k 13, max_k 127, step 6
    jobs = repeat_lib.window_jobs(20261017, args.windows, k_values=kvals, lengths=(1000,))
    scan = GpuRepeatScan(library=args.library)
    for _ in range(args.warmup):
        got, _ = scan.scan(jobs)
    t0 = time.perf_counter()
    ker = []
    for _ in range(args.steps):
        got, ms = scan.scan(jobs)
        ker.append(ms)
    wall = (time.perf_counter() - t0) / args.steps
    kms = float(np.median(ker))
    # pairs the reference would visit when nothing repeats: C(n_kmers, 2) per job
    pairs = sum((len(s) - k + 1) * (len(s) - k) // 2 for s, k, _ in jobs)
    ref = repeat_lib.reference()
    lib, kind = (ref, "reference") if ref is not None else (repeat_lib.oracle(), "port")
    fn = lib.ref_has_repeat if ref is not None else lib.orc_has_repeat
    idx = np.linspace(0, len(jobs) - 1, args.cpu_jobs).astype(int)
    t0 = time.perf_counter()
    cpu = [fn(jobs[i][0], len(jobs[i][0]), jobs[i][1], jobs[i][2]) for i in idx]
    cpu_s = time.perf_counter() - t0
    assert [int(got[i]) for i in idx] == cpu, "GPU and CPU answers differ"
    print(json.dumps({
        "metric": "repeat_jobs_per_sec", "unit": "jobs/s", "jobs": len(jobs), "windows": args.windows,
        "library": args.library or "main", "k_values": list(kvals), "window_len": "1000-1049", "repeat_fraction": round(float((got == 1).mean()), 4),
        "e2e": {"value": len(jobs) / wall, "ms_per_call": wall * 1e3, "note": "lgr_repeat_scan with host buffers"},
        "kernel": {"value": len(jobs) / (kms * 1e-3), "ms": kms, "kmer_pairs_upper_bound_per_s": pairs / (kms * 1e-3)},
        "cpu_baseline": {"value": len(idx) / cpu_s, "unit": "jobs/s", "cores": 1, "kind": kind,
                         "sample": f"{len(idx)} evenly spaced jobs of the same workload"},
    }))


if __name__ == "__main__":
    main()
