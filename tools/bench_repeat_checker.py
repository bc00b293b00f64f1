#!/usr/bin/env python
"""The repeat check in Lancet2's call pattern (DESIGN §11): worker threads that each ask about one window at a time.
Writes JSON lines (default profiles/r3_repeat_checker.jsonl), the GPU's name and power limit first:
  lone_window   latency of one window alone (1 kb and 2.5 kb, Lancet2's 20 k values with 2 mismatches plus the exact
                question at max_k) through lgr_repeat_scan, shipped build (diagonal slices) against the one-slice build
  threads       windows/s from 1, 4, 16 and 64 C++ threads: through one RepeatChecker, through one private
                lgr_repeat_scan context per thread, and through the CPU oracle (or the reference's own HasRepeat when
                built) on as many threads, on a sample of the same windows"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import repeat_lib  # noqa: E402
from lancet2_b200.repeat_scan import ONE_SLICE_LIBRARY, GpuRepeatScan, RepeatChecker, private_contexts_run  # noqa: E402

K_LOOP = tuple(range(13, 128, 6))  # Lancet2's defaults: min_k 13, max_k 127, step 6
QUESTIONS = [(k, 2) for k in K_LOOP] + [(max(K_LOOP), 0)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def windows_of(seed, n, length):
    jobs = repeat_lib.window_jobs(seed, n, k_values=K_LOOP, lengths=(length,))
    q = len(QUESTIONS)
    return [(jobs[w * q][0], QUESTIONS) for w in range(n)]


def lone_window(length, library, reps):
    scan = GpuRepeatScan(library=library)
    wins = windows_of(11 + length, 8, length)
    for s, qs in wins:  # warm-up
        scan.scan([(s, k, mm) for k, mm in qs])
    wall, ker = [], []
    for i in range(reps):
        s, qs = wins[i % len(wins)]
        t0 = time.perf_counter()
        _, ms = scan.scan([(s, k, mm) for k, mm in qs])
        wall.append((time.perf_counter() - t0) * 1e3)
        ker.append(ms)
    scan.close()
    return {"kind": "lone_window", "window_len": f"{length}-{length + 49}", "questions": len(QUESTIONS),
            "library": "one_slice" if library else "main", "calls": reps,
            "ms_per_call_median": float(np.median(wall)), "ms_per_call_p90": float(np.percentile(wall, 90)),
            "kernel_ms_median": float(np.median(ker))}


def cpu_arm(windows, threads):
    ref = repeat_lib.reference()
    lib, fn, kind = (ref, ref.ref_has_repeat, "reference") if ref is not None else \
        (repeat_lib.oracle(), repeat_lib.oracle().orc_has_repeat, "port")

    def one(w):
        s, qs = w
        return [fn(s, len(s), k, mm) for k, mm in qs]

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:  # ctypes releases the GIL inside the call
        ans = list(ex.map(one, windows))
    return len(windows) / (time.perf_counter() - t0), ans, kind


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=2000)
    ap.add_argument("--length", type=int, default=1000)
    ap.add_argument("--threads", default="1,4,16,64")
    ap.add_argument("--lone-calls", type=int, default=200)
    ap.add_argument("--cpu-windows-per-thread", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_repeat_checker.jsonl"))
    args = ap.parse_args()
    lines = [dict(kind="device", **gpu_info(), host_cpus=os.cpu_count())]
    for length in (1000, 2500):
        for library in (None, ONE_SLICE_LIBRARY):
            lines.append(lone_window(length, library, args.lone_calls))
            print(json.dumps(lines[-1]), flush=True)
    wins = windows_of(20261021, args.windows, args.length)
    for threads in [int(t) for t in args.threads.split(",")]:
        chk = RepeatChecker()
        chk.run(wins[:64], threads=min(threads, 64))  # warm-up
        chk.close()
        chk = RepeatChecker()
        got, status, ctr = chk.run(wins, threads=threads)
        chk.close()
        assert (status == 0).all()
        priv, pstatus, pns = private_contexts_run(wins, threads=threads)
        assert (pstatus == 0).all() and all(np.array_equal(a, b) for a, b in zip(got, priv))
        n_cpu = min(len(wins), max(args.cpu_windows_per_thread * threads, 8))
        idx = np.linspace(0, len(wins) - 1, n_cpu).astype(int)
        cpu_rate, cpu_ans, kind = cpu_arm([wins[i] for i in idx], threads)
        assert all(list(got[i]) == a for i, a in zip(idx, cpu_ans)), "GPU and CPU answers differ"
        lines.append({"kind": "threads", "threads": threads, "windows": len(wins), "window_len": f"{args.length}-{args.length + 49}",
                      "questions_per_window": len(QUESTIONS),
                      "checker_windows_per_s": len(wins) / (ctr["ns_wall"] * 1e-9),
                      "checker": {k: ctr[k] for k in ("batches", "max_windows_in_batch", "ns_wait", "ns_wall")},
                      "private_contexts_windows_per_s": len(wins) / (pns * 1e-9),
                      "cpu_windows_per_s": cpu_rate, "cpu_threads": threads, "cpu_kind": kind, "cpu_sample_windows": n_cpu})
        print(json.dumps(lines[-1]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
