"""The grow-only device buffer of the three CUDA libraries (lancet2_b200/csrc/lgr_host.h): an allocation the
driver refuses leaves the buffer empty, says why, and does not fail the next call on the same thread."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from compare import compare_results
from lancet2_b200 import abi, synth

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lancet2_b200", "csrc")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
LGR_E_NOMEM = -6
PETABYTE = 1 << 50  # refused by the driver at once: an error return, not a fault

_PROBE = r"""
#include "lgr_host.h"
#include <cstdio>
extern "C" int probe_ensure(unsigned long long bytes, void** p, unsigned long long* cap, char* err, int err_cap) {
  DeviceBuffer b;
  std::string e;
  const int rc = b.ensure(bytes, false, e);
  *p = b.p, *cap = b.cap;
  std::snprintf(err, err_cap, "%s", e.c_str());
  return rc;
}
"""


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    """lgr_host.h compiled by g++ against the CUDA runtime: no device code, no GPU needed to load it."""
    d = tmp_path_factory.mktemp("host_buffers")
    src, so = d / "probe.cpp", d / "libprobe.so"
    src.write_text(_PROBE)
    lib64 = os.path.join(CUDA, "lib64")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, "-I", os.path.join(CUDA, "include"),
                           "-o", str(so), str(src), "-L", lib64, "-lcudart", "-Wl,-rpath," + lib64])
    lib = C.CDLL(str(so))
    lib.probe_ensure.argtypes = [C.c_ulonglong, C.POINTER(C.c_void_p), C.POINTER(C.c_ulonglong), C.c_char_p, C.c_int]
    lib.probe_ensure.restype = C.c_int
    return lib


def test_refused_allocation_leaves_the_buffer_empty(probe):
    p, cap, err = C.c_void_p(1), C.c_ulonglong(1), C.create_string_buffer(256)
    assert probe.probe_ensure(PETABYTE, C.byref(p), C.byref(cap), err, len(err)) == LGR_E_NOMEM
    assert p.value is None and cap.value == 0
    assert err.value.startswith(b"cudaMalloc(")


# ---- after a refused reservation, the next call on the same context and thread succeeds ----

@pytest.fixture(scope="module")
def batch_and_fresh_result():
    from lancet2_b200.realign import GpuRealigner
    batch = abi.Batch(synth.make_groups(23, 4, n_reads=48, n_haps=3, hap_len=500))
    fresh = GpuRealigner(0)
    try:
        want, _ = fresh.genotype_batch(batch)
    finally:
        fresh.close()
    return batch, want


@pytest.mark.gpu
def test_batch_after_refused_lgr_reserve(batch_and_fresh_result):
    from lancet2_b200.realign import GpuRealigner
    batch, want = batch_and_fresh_result
    g = GpuRealigner(0)
    try:
        assert g.lib.lgr_reserve(g._ctx, PETABYTE, 1) == LGR_E_NOMEM
        assert g.lib.lgr_last_error(g._ctx).startswith(b"cudaMalloc(")
        got, _ = g.genotype_batch(batch)
        assert got.rc == 0
        errs = compare_results(batch, want, got)
        assert not errs, "\n".join(errs[:20])
        assert got.assign[:batch.n_assign].tobytes() == want.assign[:batch.n_assign].tobytes()
    finally:
        g.close()


@pytest.mark.gpu
def test_scan_after_refused_lgr_repeat_reserve():
    import repeat_lib
    from lancet2_b200.repeat_scan import GpuRepeatScan
    jobs = repeat_lib.window_jobs(31, 12)
    fresh = GpuRepeatScan()
    try:
        want, _ = fresh.scan(jobs)
    finally:
        fresh.close()
    scan = GpuRepeatScan()
    try:
        assert scan._lib.lgr_repeat_reserve(scan._ctx, PETABYTE, 1) == LGR_E_NOMEM
        got, _ = scan.scan(jobs)
        assert scan.last_rc == 0
        assert np.array_equal(got, want)
    finally:
        scan.close()
