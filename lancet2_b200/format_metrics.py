"""Host-side handle of the device FORMAT path (SURVEY.md §8f #2): the evidence streams of many
`caller::VariantSupport` objects in, every FORMAT accessor's value out
(reference: src/lancet/caller/variant_support.h:60-330).  Plumbing only — the arithmetic is
k_fmt_dedup / k_fmt_metrics in csrc/lgr_format.cu; there is no CPU implementation here and the
constructor raises when the CUDA library or a device is missing."""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence, Tuple

import numpy as np

from . import abi


class GpuFormatMetrics:
    def __init__(self, device: int = 0):
        self._main = abi.load_library()
        self._lib = self._main
        # A/B builds of the same four entry points (e.g. csrc/liblgr_format_scan.so, the O(n^2)-scan kernels; the shipped build is -DLGR_FMT_SORT)
        variant = os.environ.get("LGR_FORMAT_LIBRARY")
        if variant:
            self._lib = C.CDLL(variant)
            self._lib.lgr_format_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
            self._lib.lgr_format_create.restype = C.c_int
            self._lib.lgr_format_destroy.argtypes = [C.c_void_p]
            self._lib.lgr_format_destroy.restype = None
            self._lib.lgr_format_last_error.argtypes = [C.c_void_p]
            self._lib.lgr_format_last_error.restype = C.c_char_p
            self._lib.lgr_format_metrics.argtypes = [C.c_void_p, C.POINTER(abi.LgrEvidenceIn), C.c_void_p, C.POINTER(C.c_float)]
            self._lib.lgr_format_metrics.restype = C.c_int
        self._ctx = C.c_void_p()
        rc = self._lib.lgr_format_create(device, C.byref(self._ctx))
        if rc != 0:
            msg = self._lib.lgr_format_last_error(None).decode()
            self._ctx = C.c_void_p()
            raise RuntimeError(f"lgr_format_create failed ({self._main.lgr_strerror(rc).decode()}): {msg}")

    def close(self) -> None:
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.lgr_format_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def compute(self, batch: "abi.EvidenceBatch | Sequence[dict]") -> Tuple[np.ndarray, float]:
        """(records of abi.FORMAT_DTYPE, one per support; CUDA-event ms of the two kernels)."""
        if not isinstance(batch, abi.EvidenceBatch):
            batch = abi.EvidenceBatch(batch)
        out = np.zeros(batch.n_supports, dtype=abi.FORMAT_DTYPE)
        st = batch.c_struct()
        ms = C.c_float(0.0)
        rc = self._lib.lgr_format_metrics(self._ctx, C.byref(st), out.ctypes.data, C.byref(ms))
        self.last_rc = rc
        if rc == abi.LGR_E_PARTIAL:  # supports with more than LGR_FMT_MAX_ALLELES alleles are flagged, not fatal
            return out, float(ms.value)
        if rc != 0:
            raise RuntimeError(f"lgr_format_metrics failed ({self._main.lgr_strerror(rc).decode()}): "
                               f"{self._lib.lgr_format_last_error(self._ctx).decode()}")
        return out, float(ms.value)

    def compute_packed(self, windows, dir_inside: bool = True) -> Tuple[np.ndarray, float]:
        """The same records as compute() on every window's supports concatenated, through lgr_format_pack and ONE
        lgr_format_metrics_packed.  `windows`: a sequence of windows (lists of support dicts) or a PackedWindows."""
        pk = windows if isinstance(windows, PackedWindows) else PackedWindows(windows, self._main, dir_inside)
        return self.metrics_packed(pk)

    def metrics_packed(self, pk: PackedWindows, slab_ptr: int = 0) -> Tuple[np.ndarray, float]:
        """lgr_format_metrics_packed on packed windows (slab_ptr: a copy of pk.slab to send instead, e.g. pinned).
        → (records of every window's supports in directory order, CUDA-event ms of the three kernels)."""
        if self._lib is not self._main:
            raise RuntimeError("the packed path is not part of the A/B FORMAT libraries")
        out = np.zeros(max(pk.n_supports, 1), dtype=abi.FORMAT_DTYPE)
        st = pk.c_struct(slab_ptr)
        ms = C.c_float(0.0)
        rc = self._lib.lgr_format_metrics_packed(self._ctx, C.byref(st), out.ctypes.data, C.byref(ms))
        self.last_rc = rc
        if rc not in (0, abi.LGR_E_PARTIAL):
            raise RuntimeError(f"lgr_format_metrics_packed failed ({self._main.lgr_strerror(rc).decode()}): "
                               f"{self._lib.lgr_format_last_error(self._ctx).decode()}")
        return out[:pk.n_supports], float(ms.value)

    def reserve(self, slab_bytes: int, n_supports: int, n_evidence: int) -> None:
        rc = self._main.lgr_format_reserve(self._ctx, slab_bytes, n_supports, n_evidence)
        if rc != 0:
            raise RuntimeError(f"lgr_format_reserve failed: {self._main.lgr_format_last_error(self._ctx).decode()}")

    def device_bytes(self) -> int:
        """device bytes the context holds (lgr_format_device_bytes)"""
        return int(self._main.lgr_format_device_bytes(self._ctx))

    def from_assign(self, batch: "abi.Batch", *, n_samples: int, sample_id, start0, isize, sam_flag, mapq, softclip,
                    var_n_alleles, var_len, host_assign=None, dev_assign: int = 0):
        """AddToTable + FORMAT math on the device (lgr_format_from_assign): evidence columns are built by
        k_evidence_* from the realignment's lgr_assign records — `dev_assign` (a device address from
        GpuRealigner.resident_assign()) or `host_assign` (numpy records, uploaded) — and the per-read fields.
        → (records, keys[S,3] = group / variant / sample id, CUDA-event ms of all kernels)."""
        if self._lib is not self._main:
            raise RuntimeError("from_assign is not part of the A/B FORMAT libraries")
        keep = [np.ascontiguousarray(a, dtype=dt) for a, dt in (
            (batch.grp_read_begin, np.int32), (batch.grp_var_begin, np.int32),
            (np.diff(batch.grp_hap_begin), np.int32), (var_n_alleles, np.int32), (var_len, np.int32), (isize, np.int64),
            (start0, np.int64), (batch.read_name_hash, np.uint32), (sample_id, np.int32), (sam_flag, np.uint16),
            (mapq, np.uint8), (softclip, np.uint8))]
        st = abi.LgrAssignBatch()
        st.dev_assign = dev_assign or None
        if host_assign is not None:
            host_assign = np.ascontiguousarray(host_assign)
            st.host_assign = host_assign.ctypes.data
        st.n_assign = int(batch.n_assign)
        st.n_groups, st.n_reads, st.n_vars, st.n_samples = batch.n_groups, batch.n_reads, batch.n_vars, n_samples
        for name, arr in zip(("grp_read_begin", "grp_var_begin", "grp_n_haps", "var_n_alleles", "var_len", "read_insert_size",
                              "read_aln_start", "read_name_hash", "read_sample", "read_sam_flag", "read_map_qual",
                              "read_soft_clipped"), keep):
            setattr(st, name, arr.ctypes.data)
        cap = max(1, batch.n_vars * n_samples)
        out = np.zeros(cap, dtype=abi.FORMAT_DTYPE)
        keys = np.zeros((cap, 3), dtype=np.int32)
        n_sup, ms = C.c_int32(0), C.c_float(0.0)
        rc = self._lib.lgr_format_from_assign(self._ctx, C.byref(st), out.ctypes.data, cap, keys.ctypes.data, C.byref(n_sup), C.byref(ms))
        self.last_rc = rc
        if rc not in (0, abi.LGR_E_PARTIAL):
            raise RuntimeError(f"lgr_format_from_assign failed ({self._main.lgr_strerror(rc).decode()}): "
                               f"{self._lib.lgr_format_last_error(self._ctx).decode()}")
        return out[:n_sup.value], keys[:n_sup.value], float(ms.value)

    def debug_evidence(self) -> dict:
        """The evidence columns the last from_assign built on the device (test hook)."""
        probe = abi.LgrEvidenceIn()
        if self._lib.lgr_format_debug_evidence(self._ctx, C.byref(probe)) != 0:
            raise RuntimeError("lgr_format_debug_evidence failed")
        n, s = int(probe.n_evidence), int(probe.n_supports)
        cols = {"sup_begin": np.zeros(s + 1, np.int64), "sup_n_alleles": np.zeros(s, np.int32),
                "sup_variant_len": np.zeros(s, np.int32), "sup_total_haps": np.zeros(s, np.int32)}
        for name, dt in abi.EVIDENCE_FIELDS:
            cols[name] = np.zeros(n, dtype=dt)
        st = abi.LgrEvidenceIn()
        for name, arr in cols.items():
            setattr(st, name, arr.ctypes.data if arr.size else None)
        if self._lib.lgr_format_debug_evidence(self._ctx, C.byref(st)) != 0:
            raise RuntimeError("lgr_format_debug_evidence failed")
        return cols


class PackedWindows:
    """Windows (each a list of support dicts, or an abi.EvidenceBatch) packed with lgr_format_pack into one slab, the
    directory placed behind the blocks (one host->device copy) or, with dir_inside=False, in an array of its own.
    `dir` is a numpy view (abi.FMT_DIR_DTYPE) that may be edited before the call."""

    def __init__(self, windows, lib, dir_inside: bool = True):
        self.batches = [w if isinstance(w, abi.EvidenceBatch) else abi.EvidenceBatch(w) for w in windows]
        structs = [b.c_struct() for b in self.batches]
        sizes = [int(lib.lgr_format_packed_bytes(C.byref(st))) for st in structs]
        if any(n == 0 for n in sizes):
            raise ValueError("malformed window (lgr_format_packed_bytes returned 0)")
        self.rec_bytes = sum(sizes)
        n = len(structs)
        dir_bytes = n * abi.FMT_DIR_DTYPE.itemsize
        self.slab = np.zeros(self.rec_bytes + (dir_bytes if dir_inside else 0) + 16, dtype=np.uint8)
        self.slab_bytes = self.rec_bytes + (dir_bytes if dir_inside else 0)
        if dir_inside:
            self.dir = self.slab[self.rec_bytes:self.rec_bytes + dir_bytes].view(abi.FMT_DIR_DTYPE)
        else:
            self.dir = np.zeros(n, dtype=abi.FMT_DIR_DTYPE)
        off = sup = ev = 0
        d = abi.LgrFmtDir()
        for w, (st, size) in enumerate(zip(structs, sizes)):
            rc = lib.lgr_format_pack(C.byref(st), self.slab.ctypes.data + off, size, C.byref(d))
            if rc != 0:
                raise ValueError(f"lgr_format_pack refused window {w} ({rc})")
            self.dir[w] = (off, d.n_evidence, ev, d.n_supports, sup, d.n_wide, (0, 0, 0))
            off, sup, ev = off + size, sup + d.n_supports, ev + d.n_evidence
        self.n_windows, self.n_supports, self.n_evidence = n, sup, ev

    def c_struct(self, slab_ptr: int = 0) -> abi.LgrFmtPackedIn:
        """slab_ptr: the address of a copy of self.slab (e.g. pinned memory) to hand over instead"""
        st = abi.LgrFmtPackedIn()
        st.n_windows, st.slab_bytes = self.n_windows, self.slab_bytes
        st.slab = slab_ptr or self.slab.ctypes.data
        inside = self.dir.base is not None and np.shares_memory(self.dir, self.slab)
        st.dir = (st.slab + self.rec_bytes) if inside else self.dir.ctypes.data
        return st


def _bind_calculator(lib: C.CDLL) -> C.CDLL:
    lib.lgr_adapter_format_calculator_create.argtypes = [C.c_int, C.c_longlong, C.c_longlong, C.c_longlong, C.c_char_p, C.c_int]
    lib.lgr_adapter_format_calculator_create.restype = C.c_void_p
    lib.lgr_adapter_format_calculator_destroy.argtypes = [C.c_void_p]
    lib.lgr_adapter_format_calculator_destroy.restype = None
    lib.lgr_adapter_format_calculator_run.argtypes = [C.c_void_p, C.POINTER(abi.LgrEvidenceIn), C.c_void_p, C.c_int, C.c_int,
                                                      C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lgr_adapter_format_calculator_run.restype = C.c_int
    lib.lgr_adapter_format_private_run.argtypes = [C.c_int, C.POINTER(abi.LgrEvidenceIn), C.c_void_p, C.c_int, C.c_int,
                                                   C.c_void_p, C.c_void_p]
    lib.lgr_adapter_format_private_run.restype = C.c_longlong
    return lib


class _FlatWindows:
    """Windows as one flat EvidenceBatch plus the support range of each window (the adapter's run hooks)."""

    def __init__(self, windows):
        self.batch = abi.EvidenceBatch([s for w in windows for s in w])
        self.win_sup_begin = np.concatenate([[0], np.cumsum([len(w) for w in windows])]).astype(np.int32)
        self.n = len(windows)
        self.st = self.batch.c_struct()
        self.out = np.zeros(max(self.batch.n_supports, 1), dtype=abi.FORMAT_DTYPE)
        self.status = np.full(self.n + 1, -1, dtype=np.int32)

    def per_window(self):
        return [self.out[self.win_sup_begin[w]:self.win_sup_begin[w + 1]].copy() for w in range(self.n)]


class FormatCalculator:
    """Handle on the C++ lancet_gpu::FormatCalculator (host/gpu_format.h): one calculator per GPU, called from many
    C++ threads.  Construction raises without a GPU (no CPU fallback)."""

    COUNTERS = ("batches", "windows", "supports", "evidence", "max_windows_in_batch", "alone", "ns_pack", "ns_seal_wait",
                "ns_device", "ns_wall")

    def __init__(self, device: int = 0, slab_bytes: int = 0, max_supports: int = 0, max_evidence: int = 0):
        """slab_bytes / max_supports / max_evidence: the calculator's per-slab sizes (0 = its defaults)."""
        self._lib = _bind_calculator(abi.load_library())
        err = C.create_string_buffer(512)
        self._h = self._lib.lgr_adapter_format_calculator_create(device, slab_bytes, max_supports, max_evidence, err, len(err))
        if not self._h:
            raise RuntimeError(f"FormatCalculator construction failed: {err.value.decode()}")

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.lgr_adapter_format_calculator_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, windows, threads: int = 1):
        """Every window (a list of support dicts) through FormatCalculator::Compute from `threads` C++ threads (window w
        on thread w % threads).  → (records per window, status per window: 0 ok, 1 std::invalid_argument, 2 other
        exception, counters)."""
        if not self._h:
            raise RuntimeError("FormatCalculator is closed")
        fw = _FlatWindows(windows)
        ctr = (C.c_ulonglong * len(self.COUNTERS))()
        rc = self._lib.lgr_adapter_format_calculator_run(self._h, C.byref(fw.st), fw.win_sup_begin.ctypes.data, fw.n, threads,
                                                         fw.out.ctypes.data, fw.status.ctypes.data, ctr)
        if rc != 0:
            raise RuntimeError(f"lgr_adapter_format_calculator_run failed ({rc})")
        return fw.per_window(), fw.status[:fw.n].copy(), dict(zip(self.COUNTERS, list(ctr)))


def private_contexts_run(windows, threads: int = 1, device: int = 0):
    """The binding without a calculator: every C++ thread owns a FORMAT context and makes one lgr_format_metrics per
    window.  → (records per window, status per window, wall ns)."""
    lib = _bind_calculator(abi.load_library())
    fw = _FlatWindows(windows)
    ns = lib.lgr_adapter_format_private_run(device, C.byref(fw.st), fw.win_sup_begin.ctypes.data, fw.n, threads,
                                            fw.out.ctypes.data, fw.status.ctypes.data)
    if ns < 0:
        raise RuntimeError("lgr_adapter_format_private_run: no FORMAT context")
    return fw.per_window(), fw.status[:fw.n].copy(), int(ns)
