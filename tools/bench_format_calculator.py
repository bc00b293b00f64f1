#!/usr/bin/env python
"""The FORMAT row in Lancet2's call pattern (DESIGN §10): worker threads that each compute one window at a time.
Writes JSON lines (default profiles/r3_format_calculator.jsonl), the GPU's name and power limit first:
  per_call   wall ms and kernel ms of one call: lgr_format_metrics from host buffers (16 copies) against
             lgr_format_metrics_packed from a pinned slab (one copy, packed beforehand), for the supports of a cfg2 step
             (506 supports of ~230 records) and for one window's supports (3); old and new alternate, three rounds
  threads    windows/s from 1, 4, 16 and 64 C++ threads: through one FormatCalculator, and through one private
             FORMAT context per thread (lgr_format_metrics per window); every record compared between the two"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import format_lib as F  # noqa: E402
from lancet2_b200 import abi  # noqa: E402
from lancet2_b200.format_metrics import FormatCalculator, GpuFormatMetrics, PackedWindows, private_contexts_run  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def cfg2_supports(rng, n_sup):
    # the shape of tools/bench_format.py's cfg2-step: ~230 records per support, two alleles
    return [F.random_support(rng, n=int(rng.integers(184, 276)), n_alleles=2, dup_frac=0.4) for _ in range(n_sup)]


def per_call(fmt, shape, sups, windows, reps, rounds=3):
    lib = fmt._main
    batch = abi.EvidenceBatch(sups)
    st = batch.c_struct()
    out = np.zeros(len(sups), dtype=abi.FORMAT_DTYPE)
    pk = PackedWindows(windows, lib)
    pinned = lib.lgr_alloc_pinned(len(pk.slab))
    C.memmove(pinned, pk.slab.ctypes.data, len(pk.slab))
    pst = pk.c_struct(pinned)
    out2 = np.zeros(len(sups), dtype=abi.FORMAT_DTYPE)
    ms = C.c_float()
    lines = []
    for _ in range(5):  # warm-up of both shapes
        lib.lgr_format_metrics(fmt._ctx, C.byref(st), out.ctypes.data, C.byref(ms))
        lib.lgr_format_metrics_packed(fmt._ctx, C.byref(pst), out2.ctypes.data, C.byref(ms))
    assert out.tobytes() == out2.tobytes()
    for rnd in range(rounds):
        for arm in ("lgr_format_metrics", "lgr_format_metrics_packed"):
            wall, ker = [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                if arm == "lgr_format_metrics":
                    rc = lib.lgr_format_metrics(fmt._ctx, C.byref(st), out.ctypes.data, C.byref(ms))
                else:
                    rc = lib.lgr_format_metrics_packed(fmt._ctx, C.byref(pst), out2.ctypes.data, C.byref(ms))
                wall.append((time.perf_counter() - t0) * 1e3)
                ker.append(ms.value)
                assert rc == 0
            lines.append({"kind": "per_call", "shape": shape, "supports": len(sups), "records": int(batch.n_evidence),
                          "windows": len(windows), "arm": arm, "round": rnd, "calls": reps,
                          "ms_per_call_median": float(np.median(wall)), "ms_per_call_p90": float(np.percentile(wall, 90)),
                          "kernel_ms_median": float(np.median(ker))})
            print(json.dumps(lines[-1]), flush=True)
    assert out.tobytes() == out2.tobytes()
    lib.lgr_free_pinned(pinned)
    t0 = time.perf_counter()
    for _ in range(reps):
        PackedWindows(windows, lib)
    lines.append({"kind": "pack_python", "shape": shape, "ms_per_pack": (time.perf_counter() - t0) * 1e3 / reps,
                  "note": "ctypes + numpy packing of the windows in Python, for scale only"})
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--windows", type=int, default=4000)
    ap.add_argument("--threads", default="1,4,16,64")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_format_calculator.jsonl"))
    args = ap.parse_args()
    lines = [dict(kind="device", **gpu_info(), host_cpus=os.cpu_count())]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(20261022)
    fmt = GpuFormatMetrics(0)
    step = cfg2_supports(rng, 506)
    # a cfg2 step is 253 variants x 2 samples over a whole 1 Mb region: as windows, two supports (one variant) each
    lines += per_call(fmt, "cfg2-step", step, [step[i:i + 2] for i in range(0, len(step), 2)], args.reps)
    one = step[:3]
    lines += per_call(fmt, "one-window", one, [one], args.reps)
    fmt.close()
    # the threads arm: windows of 1-4 supports of the cfg2 shape
    wins = []
    for _ in range(args.windows):
        wins.append(cfg2_supports(rng, int(rng.integers(1, 5))))
    for threads in [int(t) for t in args.threads.split(",")]:
        calc = FormatCalculator()
        calc.run(wins[:128], threads=min(threads, 64))  # warm-up
        calc.close()
        calc = FormatCalculator()
        got, status, ctr = calc.run(wins, threads=threads)
        calc.close()
        assert (status == 0).all()
        priv, pstatus, pns = private_contexts_run(wins, threads=threads)
        assert (pstatus == 0).all() and all(a.tobytes() == b.tobytes() for a, b in zip(got, priv))
        lines.append({"kind": "threads", "threads": threads, "windows": len(wins),
                      "supports": int(sum(len(w) for w in wins)), "records_per_support": "184-275",
                      "calculator_windows_per_s": len(wins) / (ctr["ns_wall"] * 1e-9),
                      "calculator": {k: ctr[k] for k in ("batches", "max_windows_in_batch", "alone", "ns_pack",
                                                         "ns_seal_wait", "ns_device", "ns_wall")},
                      "private_contexts_windows_per_s": len(wins) / (pns * 1e-9)})
        print(json.dumps(lines[-1]), flush=True)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
