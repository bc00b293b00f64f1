#!/usr/bin/env python3
"""Device work counters of one pass over a workload (diagnostics): why pairs went to the cold chain
kernel, extension tasks per size class.  usage: python tools/debug_counters.py [cfg2|micro|tiny]"""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from lancet2_b200 import abi  # noqa: E402
from lancet2_b200.realign import GpuRealigner  # noqa: E402

NAMES = ["ITEM", "NTASK0", "NTASK1", "NTASK2", "NTASK3", "NTASK4", "REGS", "EXTARENA", "CIGARENA", "NOVF", "ERR", "EVALS", "ANCH", "CELLS", "CELLSFULL",
         "ALIGNED", "TASKPOS0", "TASKPOS1", "TASKPOS2", "TASKPOS3", "TASKPOS4", "FINPOS", "OVFPOS", "OVFNEED", "NCOLD", "COLDPOS", "COLD_HIGH",
         "COLD_SORT", "COLD_LONG", "LEAN_DEFER"]


def main():
    name = sys.argv[1] if len(sys.argv) > 1 else "cfg2"
    groups, desc = bench._build_replica_workload(name, 42)
    batch = abi.Batch(groups)
    gpu = GpuRealigner(0)
    gpu.lib.lgr_debug_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    gpu.lib.lgr_debug_counters.restype = C.c_int
    packed = abi.PackedBatch(groups, gpu.lib)
    gpu.upload_packed(packed)
    st = gpu.run_resident()
    buf = (C.c_longlong * 64)()
    n = gpu.lib.lgr_debug_counters(gpu._ctx, buf, 64)
    d = {NAMES[i] if i < len(NAMES) else f"c{i}": int(buf[i]) for i in range(n)}
    d["pairs"] = batch.n_pairs
    d["workload"] = desc
    d["ms"] = {"index": st.ms_k_index, "sketch": st.ms_k_sketch, "map": st.ms_k_map, "ext": st.ms_k_ext, "assign": st.ms_k_assign, "all": st.ms_kernels}
    print(json.dumps(d))


if __name__ == "__main__":
    main()
