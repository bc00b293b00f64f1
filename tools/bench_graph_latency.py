#!/usr/bin/env python
"""Graph mode of the blocking calls (lgr_set_graph_mode) against the separate launches, in one process.
Writes JSON lines (default profiles/r3_graph_latency.jsonl), the GPU's name and power limit first:
  call     one lgr_genotype_batch / lgr_genotype_packed of 1, 4 or 16 region groups (tools/latency_probe.py's
           windows), stream and graph mode alternated on one context: per-call wall time (host clock around the
           blocking call, median and p90) and the medians of the lgr_stats copy and stage times
  direct   Genotype() calls/s through GenotypeBatcher's direct path from 1, 4 and 8 C++ threads, with
           Options::direct_graph off and on, alternated"""
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

from lancet2_b200 import abi, synth  # noqa: E402
from lancet2_b200.realign import GpuRealigner  # noqa: E402

STAGES = ("ms_h2d", "ms_kernels", "ms_d2h", "ms_k_index", "ms_k_sketch", "ms_k_map", "ms_k_ext", "ms_k_assign")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clock = [x.strip() for x in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def call_arm(gpu, groups, packed, calls, repeats):
    batch = abi.Batch(groups)
    res = abi.Result(batch, 1 << 16)
    pk = abi.PackedBatch(groups, gpu.lib) if packed else None
    if pk is not None:
        import torch
        pk.pin(torch)

    def one():
        if pk is not None:
            return gpu.genotype_packed(pk, batch, result=res, want_aln=False)[1]
        return gpu.genotype_batch(batch, result=res, want_aln=False)[1]

    for graph in (False, True):  # warm-up: module loads, arena, the graph's executable
        gpu.set_graph_mode(graph)
        for _ in range(20):
            one()
    out = []
    for rep in range(repeats):
        for graph in (False, True):
            gpu.set_graph_mode(graph)
            wall, st = [], []
            for _ in range(calls):
                t0 = time.perf_counter()
                s = one()
                wall.append((time.perf_counter() - t0) * 1e3)
                st.append([getattr(s, k) for k in STAGES])
            st = np.asarray(st)
            out.append({"kind": "call", "groups": len(groups), "pairs": batch.n_pairs, "input": "packed" if packed else "plain",
                        "mode": "graph" if graph else "stream", "repeat": rep, "calls": calls,
                        "wall_ms_median": float(np.median(wall)), "wall_ms_p90": float(np.percentile(wall, 90)),
                        **{k + "_median": float(np.median(st[:, i])) for i, k in enumerate(STAGES)},
                        "kernel_launches": int(s.kernel_launches)})
            print(json.dumps(out[-1]), flush=True)
    gpu.set_graph_mode(False)
    return out


def direct_arm(lib, threads, rounds, repeats):
    lib.lgr_adapter_direct_graph_run.argtypes = [C.c_int, C.POINTER(abi.LgrBatchIn), C.c_char_p, C.c_char_p] + \
        [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_longlong]
    lib.lgr_adapter_direct_graph_run.restype = C.c_int
    groups = synth.make_region_groups(20261021, ref_len=1_000_000)
    batch = abi.Batch(groups)
    names = [nm for g in groups for nm in g.names]
    hs = np.asarray([abi.x31_hash(nm) for nm in names], dtype=np.uint64)
    cols = (np.asarray([0 if nm.startswith("n") else 1 for nm in names], dtype=np.int32), (10_000 + hs % 10_000).astype(np.int64),
            ((hs // 7 % 1000).astype(np.int64) - 500), ((hs // 3 % 2) * 0x10 + (hs // 5 % 2) * 0x2).astype(np.uint16),
            (hs // 11 % 61).astype(np.uint8), (hs // 13 % 2).astype(np.uint8))
    blob = b"\0".join(x.encode() for x in names) + b"\0"
    bi = batch.c_struct()
    err = C.create_string_buffer(4096)

    def run(n_threads, graph, n_rounds):
        ctr = np.zeros(22, dtype=np.uint64)
        rc = lib.lgr_adapter_direct_graph_run(0, C.byref(bi), blob, b"normal\0tumor\0", *[c.ctypes.data for c in cols], n_threads,
                                              n_rounds, graph, ctr.ctypes.data, err, 0)
        if rc < 0:
            raise RuntimeError(f"lgr_adapter_direct_graph_run failed ({rc})")
        return ctr

    run(8, 0, 1), run(8, 1, 1)  # warm-up
    out = []
    for t in threads:
        for rep in range(repeats):
            for graph in (0, 1):
                ctr = run(t, graph, rounds)
                calls = int(ctr[1])
                out.append({"kind": "direct", "threads": t, "direct_graph": bool(graph), "repeat": rep, "calls": calls,
                            "pairs_per_call": batch.n_pairs / len(groups), "calls_per_s": calls / (int(ctr[4]) * 1e-9),
                            "graph_launches": int(ctr[21]), "ns_submit_per_call": int(ctr[6]) / calls})
                print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=300)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--threads", default="1,4,8")
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_graph_latency.jsonl"))
    args = ap.parse_args()
    lines = [dict(kind="device", **gpu_info(), host_cpus=os.cpu_count())]
    gs = synth.make_region_groups(42, ref_len=100_000)
    gpu = GpuRealigner(0)
    for packed in (False, True):
        for n in (1, 4, 16):
            lines += call_arm(gpu, gs[:n], packed, args.calls, args.repeats)
    lines.append(dict(kind="graph_counters", **dict(zip(("instantiated", "updated", "replayed"), gpu.graph_counters()))))
    lib = gpu.lib
    gpu.close()
    lines += direct_arm(lib, [int(t) for t in args.threads.split(",")], args.rounds, args.repeats)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
