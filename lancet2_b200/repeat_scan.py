"""Host-side handle on the repeat-detection kernel (lgr_repeat_*, SURVEY.md §8f #3 first half):
`HasRepeat(SlidingView(seq, k), max_mismatches)` of the reference (src/lancet/base/repeat.cpp:348-371,
called from cbdg/graph.h:127-131 and core/variant_builder.cpp:116-117) for many (window, k) jobs in
one device call.  No CPU path exists: construction raises when the library or a GPU is missing."""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import abi


_JOB_DTYPE = np.dtype([("seq_off", "<i8"), ("seq_len", "<i4"), ("k", "<i4"), ("max_mismatches", "<i4"), ("reserved", "<i4")])
assert _JOB_DTYPE.itemsize == C.sizeof(abi.LgrRepeatJob)


# the build with every job group on one CTA (-DLGR_REPEAT_ONE_SLICE, built beside the main library), for A/B runs
ONE_SLICE_LIBRARY = os.path.join(os.path.dirname(abi.LIB_PATH), "liblgr_repeat_one_slice.so")


def _bind_repeat(path: str) -> C.CDLL:
    """The lgr_repeat_* entry points of a stand-alone build of csrc/lgr_repeat.cu."""
    if not os.path.exists(path):
        raise RuntimeError(f"repeat library {path} is missing (built by __graft_entry__.build())")
    lib = C.CDLL(path)
    main = abi.load_library()
    for name in ("lgr_repeat_create", "lgr_repeat_destroy", "lgr_repeat_last_error", "lgr_repeat_scan", "lgr_repeat_reserve"):
        f, g = getattr(lib, name), getattr(main, name)
        f.argtypes, f.restype = g.argtypes, g.restype
    return lib


class GpuRepeatScan:
    def __init__(self, device: int = 0, library: Optional[str] = None):
        """library: a stand-alone build of the same entry points (e.g. ONE_SLICE_LIBRARY) instead of the main library."""
        self._main = abi.load_library()
        self._lib = _bind_repeat(library) if library else self._main
        self._ctx = C.c_void_p()
        rc = self._lib.lgr_repeat_create(device, C.byref(self._ctx))
        if rc != 0:
            msg = self._lib.lgr_repeat_last_error(None).decode()
            self._ctx = C.c_void_p()
            raise RuntimeError(f"lgr_repeat_create failed ({self._main.lgr_strerror(rc).decode()}): {msg}")
        self.last_rc = 0

    def close(self) -> None:
        if getattr(self, "_ctx", None) and self._ctx.value:
            self._lib.lgr_repeat_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def scan(self, jobs: Sequence[Tuple[bytes, int, int]]) -> Tuple[np.ndarray, float]:
        """jobs: (sequence, k, max_mismatches).  → (uint8 answers: 0 / 1 / LGR_REPEAT_TOO_LONG, kernel ms).
        Equal sequences are uploaded once (a window is asked once per k of the graph's k-loop)."""
        offs, blobs, pos = {}, [], 0
        arr = np.zeros(max(len(jobs), 1), dtype=_JOB_DTYPE)
        seq_off = np.empty(len(jobs), dtype=np.int64)
        for i, (seq, _, _) in enumerate(jobs):
            key = id(seq) if len(seq) > 64 else seq
            at = offs.get(key)
            if at is None:
                at = offs[key] = pos
                blobs.append(seq)
                pos += len(seq)
            seq_off[i] = at
        if jobs:
            arr["seq_off"][:len(jobs)] = seq_off
            arr["seq_len"][:len(jobs)] = [len(j[0]) for j in jobs]
            arr["k"][:len(jobs)] = [j[1] for j in jobs]
            arr["max_mismatches"][:len(jobs)] = [j[2] for j in jobs]
        buf = np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8)
        out = np.zeros(max(len(jobs), 1), dtype=np.uint8)
        ms = C.c_float(0.0)
        rc = self._lib.lgr_repeat_scan(self._ctx, buf.ctypes.data, pos, arr.ctypes.data, len(jobs), out.ctypes.data, C.byref(ms))
        self.last_rc = rc
        if rc not in (0, abi.LGR_E_PARTIAL):
            raise RuntimeError(f"lgr_repeat_scan failed ({self._main.lgr_strerror(rc).decode()}): "
                               f"{self._lib.lgr_repeat_last_error(self._ctx).decode()}")
        return out[:len(jobs)], float(ms.value)


def _bind_checker(lib: C.CDLL) -> C.CDLL:
    lib.lgr_adapter_repeat_checker_create.argtypes = [C.c_int, C.c_longlong, C.c_longlong, C.c_char_p, C.c_int]
    lib.lgr_adapter_repeat_checker_create.restype = C.c_void_p
    lib.lgr_adapter_repeat_checker_destroy.argtypes = [C.c_void_p]
    lib.lgr_adapter_repeat_checker_destroy.restype = None
    windows = [C.c_void_p] * 7  # seqs, seq_off, seq_len, n_windows, q_begin, q_k, q_mm
    windows[3] = C.c_int
    lib.lgr_adapter_repeat_checker_run.argtypes = [C.c_void_p] + windows + [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lgr_adapter_repeat_checker_run.restype = C.c_int
    lib.lgr_adapter_repeat_private_run.argtypes = [C.c_int] + windows + [C.c_int, C.c_void_p, C.c_void_p]
    lib.lgr_adapter_repeat_private_run.restype = C.c_longlong
    return lib


class _Windows:
    """(sequence, [(k, max_mismatches), ...]) per window in the flat arrays of the adapter's run hooks."""

    def __init__(self, windows: Sequence[Tuple[bytes, Sequence[Tuple[int, int]]]]):
        self.n = len(windows)
        lens = [len(s) for s, _ in windows]
        self.seq_len = np.asarray(lens + [0], dtype=np.int32)
        self.seq_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        self.seqs = np.frombuffer(b"".join(s for s, _ in windows) + b"\0", dtype=np.uint8)
        self.q_begin = np.concatenate([[0], np.cumsum([len(q) for _, q in windows])]).astype(np.int32)
        qs = [x for _, q in windows for x in q]
        self.q_k = np.asarray([k for k, _ in qs] + [0], dtype=np.int32)
        self.q_mm = np.asarray([m for _, m in qs] + [0], dtype=np.int32)
        self.answers = np.zeros(int(self.q_begin[-1]) + 1, dtype=np.uint8)
        self.status = np.zeros(self.n + 1, dtype=np.int32)

    def args(self):
        return [self.seqs.ctypes.data, self.seq_off.ctypes.data, self.seq_len.ctypes.data, self.n, self.q_begin.ctypes.data,
                self.q_k.ctypes.data, self.q_mm.ctypes.data]

    def per_window(self) -> List[np.ndarray]:
        return [self.answers[self.q_begin[w]:self.q_begin[w + 1]].copy() for w in range(self.n)]


class RepeatChecker:
    """Handle on the C++ lancet_gpu::RepeatChecker (host/gpu_repeat.h): one checker per GPU, called from many C++
    threads.  Construction raises without a GPU (no CPU fallback)."""

    COUNTERS = ("batches", "windows", "questions", "max_windows_in_batch", "ns_wait", "ns_wall", "callers_at_destroy")

    def __init__(self, device: int = 0, max_seq_bytes: int = 0, max_questions: int = 0):
        """max_seq_bytes / max_questions: the checker's reserved batch size (0 = its defaults)."""
        self._lib = _bind_checker(abi.load_library())
        err = C.create_string_buffer(512)
        self._h = self._lib.lgr_adapter_repeat_checker_create(device, max_seq_bytes, max_questions, err, len(err))
        if not self._h:
            raise RuntimeError(f"RepeatChecker construction failed: {err.value.decode()}")

    def close(self) -> None:
        if getattr(self, "_h", None):
            self._lib.lgr_adapter_repeat_checker_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def run(self, windows: Sequence[Tuple[bytes, Sequence[Tuple[int, int]]]], threads: int = 1,
            destroy: bool = False) -> Tuple[List[np.ndarray], np.ndarray, Dict[str, int]]:
        """Every window through RepeatChecker::Check from `threads` C++ threads (window w on thread w % threads).
        → (answers per window: 0 / 1 / LGR_REPEAT_TOO_LONG, status per window: 0 ok, 1 std::invalid_argument,
        2 other exception, counters).  destroy: thread t asks window t only (status -1 for the windows beyond `threads`),
        and the checker is destroyed once every thread is inside Check or back from it; this handle is then closed."""
        if not self._h:
            raise RuntimeError("RepeatChecker is closed")
        w = _Windows(windows)
        ctr = (C.c_ulonglong * 7)()
        h = self._h
        if destroy:
            self._h = None
        rc = self._lib.lgr_adapter_repeat_checker_run(h, *w.args(), threads, int(destroy), w.answers.ctypes.data,
                                                      w.status.ctypes.data, ctr)
        if rc != 0:
            raise RuntimeError(f"lgr_adapter_repeat_checker_run failed ({rc})")
        return w.per_window(), w.status[:w.n].copy(), dict(zip(self.COUNTERS, list(ctr)))


def private_contexts_run(windows: Sequence[Tuple[bytes, Sequence[Tuple[int, int]]]], threads: int = 1,
                         device: int = 0) -> Tuple[List[np.ndarray], np.ndarray, int]:
    """The binding without a checker: every C++ thread owns an lgr_repeat_scan context and asks one window per call.
    → (answers per window, status per window, wall ns)."""
    lib = _bind_checker(abi.load_library())
    w = _Windows(windows)
    ns = lib.lgr_adapter_repeat_private_run(device, *w.args(), threads, w.answers.ctypes.data, w.status.ctypes.data)
    if ns < 0:
        raise RuntimeError("lgr_adapter_repeat_private_run: no repeat context")
    return w.per_window(), w.status[:w.n].copy(), int(ns)
