"""Host-side handle on the CUDA realignment library (C-ABI in include/lancet_gpu_realign.h).

`GpuRealigner` owns one `lgr_ctx` (one GPU, one stream).  It mirrors what one
`lancet::caller::Genotyper` instance does for its worker thread (reference:
src/lancet/caller/genotyper.h:213-220) but over batches of `Genotype()` payloads.
No CPU path exists: construction raises when the library or a GPU is missing.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

from . import abi


class LgrError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"lgr error {code}: {msg}")
        self.code = code


class GpuRealigner:
    def __init__(self, device: int = 0, params: Optional[abi.LgrParams] = None, lib_path: Optional[str] = None):
        self.lib = abi.load_library(lib_path)
        if self.lib.lgr_abi_version() != 2:
            raise RuntimeError("ABI version mismatch")
        if params is None:
            params = abi.LgrParams()
            self.lib.lgr_default_params(C.byref(params))
        self.params = params
        self._ctx = C.c_void_p()
        self._inflight = {}
        rc = self.lib.lgr_create(device, C.byref(params), C.byref(self._ctx))
        if rc != 0:
            raise LgrError(rc, (self.lib.lgr_last_error(None) or b"").decode() or self.lib.lgr_strerror(rc).decode())

    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.lgr_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, partial_ok: bool = False):
        if rc == abi.LGR_E_PARTIAL and partial_ok:
            return
        if rc != 0:
            raise LgrError(rc, (self.lib.lgr_last_error(self._ctx) or b"").decode() or self.lib.lgr_strerror(rc).decode())

    def hap_mid_occ(self, hap: bytes) -> int:
        out = C.c_int32(0)
        self._check(self.lib.lgr_hap_mid_occ(self._ctx, hap, len(hap), C.byref(out)))
        return out.value

    def genotype_batch(self, batch: abi.Batch, result: Optional[abi.Result] = None, want_aln: bool = True,
                       arena: int = 1 << 20, group_status: bool = False) -> Tuple[abi.Result, abi.LgrStats]:
        """H2D + kernels + D2H through `lgr_genotype_batch` (the call a Genotyper adapter makes).
        group_status: ask for lgr_batch_out::grp_status; a batch in which some groups hit a device cap
        then returns normally with `res.rc == LGR_E_PARTIAL` and the per-group codes in `res.grp_status`."""
        res = result or abi.Result(batch, arena)
        res.want_grp_status = group_status
        bi, bo = batch.c_struct(), res.c_struct()
        if not want_aln:
            bo.aln = None
            bo.cigar_inline = None
        st = abi.LgrStats()
        res.rc = self.lib.lgr_genotype_batch(self._ctx, C.byref(bi), C.byref(bo), C.byref(st))
        self._check(res.rc, partial_ok=group_status)
        return res, st

    def submit(self, batch: abi.Batch, result: Optional[abi.Result] = None, want_aln: bool = True,
               arena: int = 1 << 20) -> Tuple[int, abi.Result]:
        """`lgr_submit`: enqueue H2D + kernels + D2H of one batch and return (ticket, result buffers).
        The buffers are filled once `wait(ticket)` returns; up to LGR_MAX_INFLIGHT tickets may be open."""
        res = result or abi.Result(batch, arena)
        bi, bo = batch.c_struct(), res.c_struct()
        if not want_aln:
            bo.aln = None
            bo.cigar_inline = None
        t = C.c_int32(-1)
        self._check(self.lib.lgr_submit(self._ctx, C.byref(bi), C.byref(bo), C.byref(t)))
        self._inflight[t.value] = (batch, res, bi, bo)  # keep every host buffer alive until wait()
        return t.value, res

    def genotype_packed(self, packed: "abi.PackedBatch", batch: abi.Batch, result: Optional[abi.Result] = None,
                        want_aln: bool = True, arena: int = 1 << 20) -> Tuple[abi.Result, abi.LgrStats]:
        """the same call on the packed wire format (`batch` only sizes the result buffers)"""
        res = result or abi.Result(batch, arena)
        pi, bo = packed.c_struct(), res.c_struct()
        if not want_aln:
            bo.aln = None
            bo.cigar_inline = None
        st = abi.LgrStats()
        self._check(self.lib.lgr_genotype_packed(self._ctx, C.byref(pi), C.byref(bo), C.byref(st)))
        return res, st

    def submit_packed(self, packed: "abi.PackedBatch", batch: abi.Batch, result: Optional[abi.Result] = None,
                      want_aln: bool = True, arena: int = 1 << 20) -> Tuple[int, abi.Result]:
        res = result or abi.Result(batch, arena)
        pi, bo = packed.c_struct(), res.c_struct()
        if not want_aln:
            bo.aln = None
            bo.cigar_inline = None
        t = C.c_int32(-1)
        self._check(self.lib.lgr_submit_packed(self._ctx, C.byref(pi), C.byref(bo), C.byref(t)))
        self._inflight[t.value] = (packed, res, pi, bo)
        return t.value, res

    def upload_packed(self, packed: "abi.PackedBatch"):
        pi = packed.c_struct()
        self._check(self.lib.lgr_upload_packed(self._ctx, C.byref(pi)))

    def wait(self, ticket: int) -> abi.LgrStats:
        st = abi.LgrStats()
        try:
            self._check(self.lib.lgr_wait(self._ctx, ticket, C.byref(st)))
        finally:
            self._inflight.pop(ticket, None)
        return st

    def upload(self, batch: abi.Batch):
        bi = batch.c_struct()
        self._check(self.lib.lgr_upload(self._ctx, C.byref(bi)))

    def run_resident(self) -> abi.LgrStats:
        st = abi.LgrStats()
        self._check(self.lib.lgr_run_resident(self._ctx, C.byref(st)))
        return st

    def download(self, batch: abi.Batch, result: Optional[abi.Result] = None, arena: int = 1 << 20) -> abi.Result:
        res = result or abi.Result(batch, arena)
        bo = res.c_struct()
        self._check(self.lib.lgr_download(self._ctx, C.byref(bo)))
        return res

    def set_graph_mode(self, on: bool = True):
        """`lgr_set_graph_mode`: run the device pass of genotype_batch / genotype_packed / run_resident as one CUDA
        graph (same results); submit / submit_packed are unaffected."""
        self._check(self.lib.lgr_set_graph_mode(self._ctx, 1 if on else 0))

    def graph_counters(self) -> Tuple[int, int, int]:
        """(instantiated, updated, replayed) executables of graph mode since the context was created"""
        i, u, r = C.c_int64(0), C.c_int64(0), C.c_int64(0)
        self._check(self.lib.lgr_graph_counters(self._ctx, C.byref(i), C.byref(u), C.byref(r)))
        return int(i.value), int(u.value), int(r.value)

    def resident_assign(self):
        """(device address, count) of the lgr_assign records of the batch this context ran last: the input of
        GpuFormatMetrics.from_assign(dev_assign=...), so the assignments never visit the host."""
        p, n = C.c_void_p(), C.c_int64(0)
        self._check(self.lib.lgr_resident_assign(self._ctx, C.byref(p), C.byref(n)))
        return int(p.value or 0), int(n.value)

    @property
    def stream(self) -> int:
        return int(self.lib.lgr_stream(self._ctx) or 0)
