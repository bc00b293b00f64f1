"""ctypes mirror of include/lancet_gpu_realign.h (the C-ABI of the realignment path).

Only plumbing lives here: struct layouts, numpy-backed batch buffers and the
loader of the CUDA library.  There is no CPU implementation in this package —
`load_library()` raises if the CUDA extension has not been built.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import numpy as np

LGR_CIGAR_INLINE = 8
LGR_MAX_READ_LEN = 1024
LGR_MAX_HAP_LEN = 65535
LGR_MAX_INFLIGHT = 4
LGR_E_LIMIT, LGR_E_PARTIAL = -4, -8

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "liblancet_gpu_realign.so")


class LgrParams(C.Structure):
    _fields_ = [
        ("k", C.c_int32), ("w", C.c_int32),
        ("a", C.c_int32), ("b", C.c_int32), ("q", C.c_int32), ("e", C.c_int32),
        ("sc_ambi", C.c_int32), ("bw", C.c_int32), ("zdrop", C.c_int32), ("end_bonus", C.c_int32),
        ("max_gap", C.c_int32), ("max_gap_ref", C.c_int32),
        ("max_chain_skip", C.c_int32), ("max_chain_iter", C.c_int32),
        ("min_cnt", C.c_int32), ("min_chain_score", C.c_int32), ("min_dp_max", C.c_int32),
        ("mid_occ", C.c_int32), ("min_mid_occ", C.c_int32), ("max_mid_occ", C.c_int32),
        ("max_max_occ", C.c_int32), ("occ_dist", C.c_int32), ("best_n", C.c_int32), ("seed", C.c_int32),
        ("mid_occ_frac", C.c_float), ("q_occ_frac", C.c_float),
        ("chain_gap_scale", C.c_float), ("chain_skip_scale", C.c_float),
        ("mask_level", C.c_float), ("pri_ratio", C.c_float), ("max_clip_ratio", C.c_float),
        ("mask_len", C.c_int32), ("cigar_arena_ops", C.c_int32),
        ("reserved", C.c_int32 * 7),
    ]


class LgrBatchIn(C.Structure):
    _fields_ = [
        ("n_groups", C.c_int32), ("n_haps", C.c_int32), ("n_reads", C.c_int32), ("n_vars", C.c_int32),
        ("grp_hap_begin", C.c_void_p), ("grp_read_begin", C.c_void_p), ("grp_var_begin", C.c_void_p),
        ("hap_off", C.c_void_p), ("hap_bases", C.c_void_p),
        ("read_off", C.c_void_p), ("read_bases", C.c_void_p), ("read_quals", C.c_void_p),
        ("read_name_hash", C.c_void_p),
        ("var_hap_off", C.c_void_p), ("var_start", C.c_void_p), ("var_len", C.c_void_p),
        ("var_allele", C.c_void_p), ("grp_mid_occ", C.c_void_p),
    ]


class LgrBatchOut(C.Structure):
    _fields_ = [
        ("n_pairs", C.c_int64), ("n_assign", C.c_int64),
        ("aln", C.c_void_p), ("cigar_inline", C.c_void_p), ("cigar_arena", C.c_void_p),
        ("cigar_arena_cap", C.c_int64), ("cigar_arena_used", C.c_int64),
        ("assign", C.c_void_p), ("grp_status", C.c_void_p), ("grp_mid_occ", C.c_void_p),
    ]


class LgrGroupDesc(C.Structure):
    _fields_ = [
        ("n_haps", C.c_int32), ("n_reads", C.c_int32), ("n_vars", C.c_int32), ("mid_occ", C.c_int32),
        ("hap_seq", C.c_void_p), ("hap_len", C.c_void_p),
        ("read_seq", C.c_void_p), ("read_qual", C.c_void_p), ("read_len", C.c_void_p),
        ("read_name_hash", C.c_void_p),
        ("var_start", C.c_void_p), ("var_len", C.c_void_p), ("var_allele", C.c_void_p),
    ]


class LgrGroupDir(C.Structure):
    _fields_ = [
        ("rec_off", C.c_uint64), ("n_haps", C.c_int32), ("n_reads", C.c_int32), ("n_vars", C.c_int32),
        ("hap_bases", C.c_int32), ("read_bases", C.c_int32), ("mid_occ", C.c_int32),
        ("max_hap_len", C.c_int32), ("max_read_len", C.c_int32),
    ]


class LgrGroupRecHdr(C.Structure):
    _fields_ = [
        ("magic", C.c_uint32), ("qual_bits", C.c_uint32), ("n_exc", C.c_uint32), ("rec_bytes", C.c_uint32),
        ("qual_lut", C.c_uint8 * 16),
        ("off_hap_len", C.c_uint32), ("off_read_len", C.c_uint32), ("off_name_hash", C.c_uint32), ("off_var", C.c_uint32),
        ("off_hap_planes", C.c_uint32), ("off_read_planes", C.c_uint32), ("off_qual", C.c_uint32), ("off_exc", C.c_uint32),
    ]


class LgrPackedIn(C.Structure):
    _fields_ = [("n_groups", C.c_int32), ("reserved", C.c_int32), ("slab", C.c_void_p), ("slab_bytes", C.c_size_t),
                ("dir", C.c_void_p)]


LGR_PACK_MAGIC = 0x3252474C
assert C.sizeof(LgrGroupDir) == 40 and C.sizeof(LgrGroupRecHdr) == 64


class LgrStats(C.Structure):
    _fields_ = [
        ("ms_h2d", C.c_float), ("ms_kernels", C.c_float), ("ms_d2h", C.c_float),
        ("ms_k_index", C.c_float), ("ms_k_sketch", C.c_float), ("ms_k_map", C.c_float),
        ("ms_k_ext", C.c_float), ("ms_k_assign", C.c_float),
        ("n_pairs", C.c_int64), ("n_aligned", C.c_int64),
        ("dp_cells", C.c_int64), ("dp_cells_full", C.c_int64),
        ("chain_evals", C.c_int64), ("n_anchors", C.c_int64),
        ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
        ("kernel_launches", C.c_int32), ("reserved", C.c_int32),
    ]


ALN_DTYPE = np.dtype([
    ("valid", "<i4"), ("score", "<i4"), ("rs", "<i4"), ("re", "<i4"), ("qs", "<i4"), ("qe", "<i4"),
    ("rev", "<i4"), ("dp_score", "<i4"), ("dp_max", "<i4"), ("mlen", "<i4"), ("blen", "<i4"),
    ("n_ambi", "<i4"), ("nm", "<i4"), ("n_cigar", "<i4"), ("cigar_off", "<i4"), ("n_regs", "<i4"),
])
assert ALN_DTYPE.itemsize == 64

ASSIGN_DTYPE = np.dtype([
    ("local_score", "<f8"), ("local_identity", "<f8"), ("folded_read_pos", "<f8"),
    ("global_score", "<i4"), ("ref_nm", "<u4"), ("own_hap_nm", "<u4"), ("hap_id", "<u4"),
    ("allele", "i1"), ("base_qual", "u1"), ("assigned", "u1"), ("pad", "u1", (5,)),
])
assert ASSIGN_DTYPE.itemsize == 48


def x31_hash(name: str) -> int:
    """minimap2 khash.h __ac_X31_hash_string (read-name hash mixed into mm_map's hit sort)."""
    b = name.encode()
    if not b:
        return 0
    h = b[0] if b[0] < 128 else b[0] - 256
    h &= 0xFFFFFFFF
    for ch in b[1:]:
        c = ch if ch < 128 else ch - 256
        h = ((h << 5) - h + c) & 0xFFFFFFFF
    return h


@dataclass
class Group:
    """Payload of one `Genotyper::Genotype(haps, reads, variant_set)` call
    (reference: src/lancet/caller/genotyper.cpp:224-235)."""
    haps: List[bytes]
    reads: List[bytes]
    quals: List[bytes]
    names: List[str]
    # per variant: list over haplotypes of (start, len, allele) with allele = -1 when absent
    variants: List[List[tuple]] = field(default_factory=list)
    mid_occ: int = 0
    # optional: index of each read's sample (ReadCollector order; AddToTable keys evidence by sample name)
    sample: Optional[List[int]] = None


class Batch:
    """Host-side SoA batch (numpy arrays) + the ctypes struct pointing at them."""

    def __init__(self, groups: Sequence[Group]):
        G = len(groups)
        ghb, grb, gvb = [0], [0], [0]
        hap_off, read_off, var_hap_off = [0], [0], [0]
        hap_chunks, read_chunks, qual_chunks = [], [], []
        name_hash, vstart, vlen, vallele = [], [], [], []
        mid = []
        pair_off, asg_off = [], []
        po = ao = 0
        for g in groups:
            P, V = len(g.haps), len(g.variants)
            for h in g.haps:
                hap_chunks.append(h)
                hap_off.append(hap_off[-1] + len(h))
            for r, q, nm in zip(g.reads, g.quals, g.names):
                assert len(r) == len(q)
                read_chunks.append(r)
                qual_chunks.append(q)
                read_off.append(read_off[-1] + len(r))
                name_hash.append(x31_hash(nm))
                pair_off.append(po)
                asg_off.append(ao)
                po += P
                ao += V
            for var in g.variants:
                assert len(var) == P
                for (s, l, a) in var:
                    vstart.append(s)
                    vlen.append(l)
                    vallele.append(a)
                var_hap_off.append(var_hap_off[-1] + P)
            ghb.append(ghb[-1] + P)
            grb.append(grb[-1] + len(g.reads))
            gvb.append(gvb[-1] + V)
            mid.append(g.mid_occ)
        pair_off.append(po)
        asg_off.append(ao)
        self.n_groups = G
        self.grp_hap_begin = np.asarray(ghb, dtype=np.int32)
        self.grp_read_begin = np.asarray(grb, dtype=np.int32)
        self.grp_var_begin = np.asarray(gvb, dtype=np.int32)
        self.hap_off = np.asarray(hap_off, dtype=np.int64)
        self.hap_bases = np.frombuffer(b"".join(hap_chunks) + b"\0", dtype=np.uint8).copy()
        self.read_off = np.asarray(read_off, dtype=np.int64)
        self.read_bases = np.frombuffer(b"".join(read_chunks) + b"\0", dtype=np.uint8).copy()
        self.read_quals = np.frombuffer(b"".join(qual_chunks) + b"\0", dtype=np.uint8).copy()
        self.read_name_hash = np.asarray(name_hash + [0], dtype=np.uint32)
        self.var_hap_off = np.asarray(var_hap_off, dtype=np.int64)
        self.var_start = np.asarray(vstart + [0], dtype=np.int32)
        self.var_len = np.asarray(vlen + [0], dtype=np.int32)
        self.var_allele = np.asarray(vallele + [0], dtype=np.int8)
        self.grp_mid_occ = np.asarray(mid + [0], dtype=np.int32)
        self.use_grp_mid_occ = any(m > 0 for m in mid)
        self.pair_off = np.asarray(pair_off, dtype=np.int64)
        self.asg_off = np.asarray(asg_off, dtype=np.int64)
        self.n_haps = int(ghb[-1])
        self.n_reads = int(grb[-1])
        self.n_vars = int(gvb[-1])
        self.n_pairs = po
        self.n_assign = ao

    def c_struct(self) -> LgrBatchIn:
        s = LgrBatchIn()
        s.n_groups, s.n_haps, s.n_reads, s.n_vars = self.n_groups, self.n_haps, self.n_reads, self.n_vars
        for name in ("grp_hap_begin", "grp_read_begin", "grp_var_begin", "hap_off", "hap_bases", "read_off",
                     "read_bases", "read_quals", "read_name_hash", "var_hap_off", "var_start", "var_len",
                     "var_allele"):
            setattr(s, name, getattr(self, name).ctypes.data)
        s.grp_mid_occ = self.grp_mid_occ.ctypes.data if self.use_grp_mid_occ else None
        return s

    def host_bytes(self) -> int:
        """bytes the C-ABI call copies host→device for this batch"""
        names = ("grp_hap_begin", "grp_read_begin", "grp_var_begin", "hap_off", "read_off", "read_name_hash",
                 "var_hap_off", "var_start", "var_len", "var_allele")
        n = sum(getattr(self, k).nbytes for k in names)
        n += int(self.hap_off[-1]) + 2 * int(self.read_off[-1])
        return n


class Result:
    """Output buffers for one batch (numpy-backed)."""

    def __init__(self, batch: Batch, cigar_arena_ops: int = 1 << 20):
        self.aln = np.zeros(max(batch.n_pairs, 1), dtype=ALN_DTYPE)
        self.cigar_inline = np.zeros(max(batch.n_pairs, 1) * LGR_CIGAR_INLINE, dtype=np.uint32)
        self.cigar_arena = np.zeros(max(cigar_arena_ops, 1), dtype=np.uint32)
        self.assign = np.zeros(max(batch.n_assign, 1), dtype=ASSIGN_DTYPE)
        self.grp_status = np.zeros(max(batch.n_groups, 1), dtype=np.int32)
        self.grp_mid_occ = np.zeros(max(batch.n_groups, 1), dtype=np.int32)
        self.want_grp_status = False
        self.n_pairs = batch.n_pairs
        self.n_assign = batch.n_assign
        self._s = LgrBatchOut()

    def c_struct(self) -> LgrBatchOut:
        s = self._s
        s.n_pairs, s.n_assign = self.n_pairs, self.n_assign
        s.aln = self.aln.ctypes.data
        s.cigar_inline = self.cigar_inline.ctypes.data
        s.cigar_arena = self.cigar_arena.ctypes.data
        s.cigar_arena_cap = self.cigar_arena.size
        s.cigar_arena_used = 0
        s.assign = self.assign.ctypes.data
        s.grp_status = self.grp_status.ctypes.data if self.want_grp_status else None
        s.grp_mid_occ = self.grp_mid_occ.ctypes.data
        return s

    def cigar(self, pair: int) -> List[int]:
        a = self.aln[pair]
        n = int(a["n_cigar"])
        if int(a["cigar_off"]) < 0:
            base = pair * LGR_CIGAR_INLINE
            return [int(x) for x in self.cigar_inline[base:base + n]]
        off = int(a["cigar_off"])
        return [int(x) for x in self.cigar_arena[off:off + n]]

    def cigar_string(self, pair: int) -> str:
        return "".join(f"{c >> 4}{'MIDNSHP=XB'[c & 0xf]}" for c in self.cigar(pair))

    def bytes_d2h(self) -> int:
        return self.n_pairs * (ALN_DTYPE.itemsize + 4 * LGR_CIGAR_INLINE) + self.n_assign * ASSIGN_DTYPE.itemsize


class PackedBatch:
    """The same groups in the packed wire format (include/lancet_gpu_realign.h): one slab of group
    records followed by the directory, built with the library's own lgr_pack_group.  `pin(torch)`
    moves the slab into page-locked memory."""

    def __init__(self, groups: Sequence[Group], lib: Optional[C.CDLL] = None):
        lib = lib or load_library()
        self.n_groups = len(groups)
        descs, keep, sizes = [], [], []
        for g in groups:
            P, R, V = len(g.haps), len(g.reads), len(g.variants)
            d = LgrGroupDesc()
            d.n_haps, d.n_reads, d.n_vars, d.mid_occ = P, R, V, int(g.mid_occ)
            hap_ptrs = (C.c_char_p * max(P, 1))(*g.haps)
            hap_len = np.asarray([len(h) for h in g.haps], dtype=np.int32)
            read_ptrs = (C.c_char_p * max(R, 1))(*g.reads)
            qual_ptrs = (C.c_char_p * max(R, 1))(*g.quals)
            read_len = np.asarray([len(r) for r in g.reads], dtype=np.int32)
            hashes = np.asarray([x31_hash(nm) for nm in g.names], dtype=np.uint32)
            vs = np.asarray([x[0] for var in g.variants for x in var], dtype=np.int32)
            vl = np.asarray([x[1] for var in g.variants for x in var], dtype=np.int32)
            va = np.asarray([x[2] for var in g.variants for x in var], dtype=np.int8)
            d.hap_seq, d.hap_len = C.cast(hap_ptrs, C.c_void_p), hap_len.ctypes.data
            d.read_seq, d.read_qual = C.cast(read_ptrs, C.c_void_p), C.cast(qual_ptrs, C.c_void_p)
            d.read_len, d.read_name_hash = read_len.ctypes.data, hashes.ctypes.data
            d.var_start, d.var_len, d.var_allele = vs.ctypes.data, vl.ctypes.data, va.ctypes.data
            keep.append((hap_ptrs, hap_len, read_ptrs, qual_ptrs, read_len, hashes, vs, vl, va))
            n = lib.lgr_packed_group_bytes(C.byref(d))
            if n == 0:
                raise ValueError("lgr_packed_group_bytes rejected a group")
            descs.append(d)
            sizes.append(n)
        rec_bytes = sum(sizes)
        self.dir = (LgrGroupDir * max(self.n_groups, 1))()
        total = rec_bytes + C.sizeof(LgrGroupDir) * self.n_groups
        self.slab = np.zeros(max(total, 16), dtype=np.uint8)
        off = 0
        for i, (d, n) in enumerate(zip(descs, sizes)):
            rc = lib.lgr_pack_group(C.byref(d), self.slab.ctypes.data + off, n, C.byref(self.dir[i]))
            if rc != 0:
                raise ValueError(f"lgr_pack_group failed with {rc}")
            self.dir[i].rec_off = off
            off += n
        self.rec_bytes = rec_bytes
        self.slab_bytes = total
        self._place_dir()

    def _place_dir(self):
        if self.n_groups:
            C.memmove(self.slab.ctypes.data + self.rec_bytes, C.addressof(self.dir), C.sizeof(LgrGroupDir) * self.n_groups)

    def pin(self, torch):
        t = torch.from_numpy(self.slab).pin_memory()
        self._pinned = t
        self.slab = t.numpy()

    def c_struct(self) -> LgrPackedIn:
        s = LgrPackedIn()
        s.n_groups = self.n_groups
        s.slab = self.slab.ctypes.data
        s.slab_bytes = self.slab_bytes
        s.dir = self.slab.ctypes.data + self.rec_bytes  # the directory copy inside the slab: ONE host->device copy
        return s


# ---- SURVEY.md §8f #2: VariantSupport aggregation + FORMAT math (lgr_format_*) ----
LGR_FMT_MAX_ALLELES = 8
LGR_FMT_MAX_GENOTYPES = 36
LGR_EV_REV, LGR_EV_SOFTCLIP, LGR_EV_PROPER_PAIR = 1, 2, 4
LGR_FMT_WIDE = 256
LGR_FMT_HAS = {"fld": 1, "mqcd": 2, "rpcd": 4, "bqcd": 8, "asmd": 16, "fsse": 32, "ahdd": 64, "hse": 128}

# SoA columns of VariantSupport::ReadEvidence (variant_support.h:64-84), in lgr_evidence_in's order
EVIDENCE_FIELDS = [("insert_size", np.int64), ("aln_start", np.int64), ("aln_score", np.float64),
                   ("folded_pos", np.float64), ("rname_hash", np.uint32), ("ref_nm", np.uint32),
                   ("own_hap_nm", np.uint32), ("hap_id", np.uint32), ("allele", np.uint8), ("flags", np.uint8),
                   ("base_qual", np.uint8), ("map_qual", np.uint8)]


class LgrEvidenceIn(C.Structure):
    _fields_ = [("n_supports", C.c_int32), ("reserved", C.c_int32), ("n_evidence", C.c_int64),
                ("sup_begin", C.c_void_p), ("sup_n_alleles", C.c_void_p), ("sup_variant_len", C.c_void_p),
                ("sup_total_haps", C.c_void_p)] + [(name, C.c_void_p) for name, _ in EVIDENCE_FIELDS]


class LgrAssignBatch(C.Structure):
    _fields_ = [("dev_assign", C.c_void_p), ("host_assign", C.c_void_p), ("n_assign", C.c_int64),
                ("n_groups", C.c_int32), ("n_reads", C.c_int32), ("n_vars", C.c_int32), ("n_samples", C.c_int32),
                ("grp_read_begin", C.c_void_p), ("grp_var_begin", C.c_void_p), ("grp_n_haps", C.c_void_p),
                ("var_n_alleles", C.c_void_p), ("var_len", C.c_void_p), ("read_insert_size", C.c_void_p),
                ("read_aln_start", C.c_void_p), ("read_name_hash", C.c_void_p), ("read_sample", C.c_void_p),
                ("read_sam_flag", C.c_void_p), ("read_map_qual", C.c_void_p), ("read_soft_clipped", C.c_void_p)]


# numpy view of lgr_format (one record per support)
FORMAT_DTYPE = np.dtype([
    ("raw_pbq", np.float64, (LGR_FMT_MAX_ALLELES,)), ("rms_mq", np.float64, (LGR_FMT_MAX_ALLELES,)),
    ("mean_aln", np.float64, (LGR_FMT_MAX_ALLELES,)), ("cmlod", np.float64, (LGR_FMT_MAX_ALLELES,)),
    ("sb", np.float64), ("sca", np.float64), ("fld", np.float64), ("mqcd", np.float64), ("rpcd", np.float64),
    ("bqcd", np.float64), ("asmd", np.float64), ("fsse", np.float64), ("ahdd", np.float64), ("hse", np.float64),
    ("fwd", np.uint32, (LGR_FMT_MAX_ALLELES,)), ("rev", np.uint32, (LGR_FMT_MAX_ALLELES,)),
    ("soft_clip", np.uint32, (LGR_FMT_MAX_ALLELES,)), ("pl", np.uint32, (LGR_FMT_MAX_GENOTYPES,)),
    ("gq", np.uint32), ("n_alleles", np.uint32), ("valid", np.uint32), ("n_kept", np.uint32)], align=True)


class EvidenceBatch:
    """S supports (one VariantSupport each) packed into the C-ABI's SoA layout.  `supports` is a
    list of dicts: the EVIDENCE_FIELDS columns (equal lengths) plus n_alleles, variant_len, total_haps."""

    def __init__(self, supports: Sequence[dict]):
        self.n_supports = len(supports)
        lens = [len(s["allele"]) for s in supports]
        self.sup_begin = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        self.n_evidence = int(self.sup_begin[-1])
        self.sup_n_alleles = np.asarray([s["n_alleles"] for s in supports], dtype=np.int32)
        self.sup_variant_len = np.asarray([s.get("variant_len", 0) for s in supports], dtype=np.int32)
        self.sup_total_haps = np.asarray([s.get("total_haps", 2) for s in supports], dtype=np.int32)
        self.cols = {}
        for name, dt in EVIDENCE_FIELDS:
            parts = [np.asarray(s[name], dtype=dt) for s in supports]
            self.cols[name] = np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(0, dt), dtype=dt)
            if len(self.cols[name]) != self.n_evidence:
                raise ValueError(f"evidence column {name} has the wrong length")

    def c_struct(self) -> LgrEvidenceIn:
        st = LgrEvidenceIn()
        st.n_supports, st.n_evidence = self.n_supports, self.n_evidence
        for name in ("sup_begin", "sup_n_alleles", "sup_variant_len", "sup_total_haps"):
            setattr(st, name, getattr(self, name).ctypes.data)
        for name, _ in EVIDENCE_FIELDS:
            setattr(st, name, self.cols[name].ctypes.data)
        return st


# packed evidence: one block per window (lgr_format_pack / lgr_format_metrics_packed)
LGR_FMT_MAGIC = 0x31544D46
LGR_FMT_SECTIONS = 16
# the sections of a block, in order: (name, element dtype, per support (+1 for sup_begin) or per record)
FMT_SECTIONS = [("sup_begin", np.int64, "S+1")] + [(n, d, "N") for n, d in EVIDENCE_FIELDS[:4]] + \
    [("sup_n_alleles", np.int32, "S"), ("sup_variant_len", np.int32, "S"), ("sup_total_haps", np.int32, "S")] + \
    [(n, d, "N") for n, d in EVIDENCE_FIELDS[4:]]


class LgrFmtBlkHdr(C.Structure):
    _fields_ = [("magic", C.c_uint32), ("n_supports", C.c_int32), ("n_evidence", C.c_int64), ("rec_bytes", C.c_uint64),
                ("reserved", C.c_uint64), ("off", C.c_uint64 * LGR_FMT_SECTIONS)]


class LgrFmtDir(C.Structure):
    _fields_ = [("rec_off", C.c_uint64), ("n_evidence", C.c_int64), ("ev_base", C.c_int64), ("n_supports", C.c_int32),
                ("sup_base", C.c_int32), ("n_wide", C.c_int32), ("reserved", C.c_int32 * 3)]


FMT_DIR_DTYPE = np.dtype([("rec_off", "<u8"), ("n_evidence", "<i8"), ("ev_base", "<i8"), ("n_supports", "<i4"),
                          ("sup_base", "<i4"), ("n_wide", "<i4"), ("reserved", "<i4", (3,))])
assert FMT_DIR_DTYPE.itemsize == C.sizeof(LgrFmtDir) == 48 and C.sizeof(LgrFmtBlkHdr) == 160


class LgrFmtPackedIn(C.Structure):
    _fields_ = [("n_windows", C.c_int32), ("reserved", C.c_int32), ("slab", C.c_void_p), ("slab_bytes", C.c_size_t),
                ("dir", C.c_void_p)]


class LgrRepeatJob(C.Structure):
    _fields_ = [("seq_off", C.c_int64), ("seq_len", C.c_int32), ("k", C.c_int32), ("max_mismatches", C.c_int32),
                ("reserved", C.c_int32)]


LGR_REPEAT_MAX_LEN = 8192
LGR_REPEAT_TOO_LONG = 255

_SYMBOLS = [
    "lgr_abi_version", "lgr_default_params", "lgr_strerror", "lgr_last_error", "lgr_x31_hash",
    "lgr_pair_offsets", "lgr_create", "lgr_destroy", "lgr_hap_mid_occ", "lgr_genotype_batch",
    "lgr_upload", "lgr_run_resident", "lgr_download", "lgr_stream", "lgr_submit", "lgr_wait",
    "lgr_alloc_pinned", "lgr_free_pinned",
    "lgr_set_notify", "lgr_set_graph_mode", "lgr_graph_counters", "lgr_reserve", "lgr_arena_bytes", "lgr_check_limits", "lgr_packed_group_bytes", "lgr_pack_group", "lgr_genotype_packed", "lgr_submit_packed", "lgr_upload_packed",
    "lgr_format_create", "lgr_format_destroy", "lgr_format_last_error", "lgr_format_metrics",
    "lgr_format_from_assign", "lgr_resident_assign", "lgr_format_debug_evidence",
    "lgr_format_packed_bytes", "lgr_format_pack", "lgr_format_metrics_packed", "lgr_format_reserve", "lgr_format_device_bytes",
    "lgr_repeat_create", "lgr_repeat_destroy", "lgr_repeat_last_error", "lgr_repeat_scan", "lgr_repeat_reserve",
]


def declared_symbols() -> List[str]:
    return list(_SYMBOLS)


def load_library(path: Optional[str] = None) -> C.CDLL:
    """dlopen the CUDA library.  Raises (never falls back) when it is missing."""
    path = path or os.environ.get("LGR_LIBRARY") or LIB_PATH  # LGR_LIBRARY: A/B builds of the same ABI
    if not os.path.exists(path):
        raise RuntimeError(
            f"CUDA extension not built: {path} is missing. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for this path).")
    lib = C.CDLL(path)
    lib.lgr_abi_version.restype = C.c_int
    lib.lgr_default_params.argtypes = [C.POINTER(LgrParams)]
    lib.lgr_default_params.restype = None
    lib.lgr_strerror.argtypes = [C.c_int]
    lib.lgr_strerror.restype = C.c_char_p
    lib.lgr_last_error.argtypes = [C.c_void_p]
    lib.lgr_last_error.restype = C.c_char_p
    lib.lgr_x31_hash.argtypes = [C.c_char_p]
    lib.lgr_x31_hash.restype = C.c_uint32
    lib.lgr_pair_offsets.argtypes = [C.POINTER(LgrBatchIn), C.c_void_p, C.c_void_p]
    lib.lgr_pair_offsets.restype = C.c_int
    lib.lgr_create.argtypes = [C.c_int, C.POINTER(LgrParams), C.POINTER(C.c_void_p)]
    lib.lgr_create.restype = C.c_int
    lib.lgr_destroy.argtypes = [C.c_void_p]
    lib.lgr_destroy.restype = None
    lib.lgr_hap_mid_occ.argtypes = [C.c_void_p, C.c_char_p, C.c_int32, C.POINTER(C.c_int32)]
    lib.lgr_hap_mid_occ.restype = C.c_int
    lib.lgr_genotype_batch.argtypes = [C.c_void_p, C.POINTER(LgrBatchIn), C.POINTER(LgrBatchOut), C.POINTER(LgrStats)]
    lib.lgr_genotype_batch.restype = C.c_int
    lib.lgr_upload.argtypes = [C.c_void_p, C.POINTER(LgrBatchIn)]
    lib.lgr_upload.restype = C.c_int
    lib.lgr_run_resident.argtypes = [C.c_void_p, C.POINTER(LgrStats)]
    lib.lgr_run_resident.restype = C.c_int
    lib.lgr_download.argtypes = [C.c_void_p, C.POINTER(LgrBatchOut)]
    lib.lgr_download.restype = C.c_int
    lib.lgr_submit.argtypes = [C.c_void_p, C.POINTER(LgrBatchIn), C.POINTER(LgrBatchOut), C.POINTER(C.c_int32)]
    lib.lgr_submit.restype = C.c_int
    lib.lgr_wait.argtypes = [C.c_void_p, C.c_int32, C.POINTER(LgrStats)]
    lib.lgr_wait.restype = C.c_int
    lib.lgr_alloc_pinned.argtypes = [C.c_size_t]
    lib.lgr_alloc_pinned.restype = C.c_void_p
    lib.lgr_free_pinned.argtypes = [C.c_void_p]
    lib.lgr_free_pinned.restype = None
    lib.lgr_set_notify.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.lgr_set_notify.restype = C.c_int
    lib.lgr_set_graph_mode.argtypes = [C.c_void_p, C.c_int]
    lib.lgr_set_graph_mode.restype = C.c_int
    lib.lgr_graph_counters.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    lib.lgr_graph_counters.restype = C.c_int
    lib.lgr_reserve.argtypes = [C.c_void_p, C.c_int64, C.c_int]
    lib.lgr_reserve.restype = C.c_int
    lib.lgr_arena_bytes.argtypes = [C.c_void_p]
    lib.lgr_arena_bytes.restype = C.c_int64
    lib.lgr_check_limits.argtypes = [C.POINTER(LgrParams), C.c_int32, C.c_int32]
    lib.lgr_check_limits.restype = C.c_int
    lib.lgr_packed_group_bytes.argtypes = [C.POINTER(LgrGroupDesc)]
    lib.lgr_packed_group_bytes.restype = C.c_size_t
    lib.lgr_pack_group.argtypes = [C.POINTER(LgrGroupDesc), C.c_void_p, C.c_size_t, C.POINTER(LgrGroupDir)]
    lib.lgr_pack_group.restype = C.c_int
    lib.lgr_genotype_packed.argtypes = [C.c_void_p, C.POINTER(LgrPackedIn), C.POINTER(LgrBatchOut), C.POINTER(LgrStats)]
    lib.lgr_genotype_packed.restype = C.c_int
    lib.lgr_submit_packed.argtypes = [C.c_void_p, C.POINTER(LgrPackedIn), C.POINTER(LgrBatchOut), C.POINTER(C.c_int32)]
    lib.lgr_submit_packed.restype = C.c_int
    lib.lgr_upload_packed.argtypes = [C.c_void_p, C.POINTER(LgrPackedIn)]
    lib.lgr_upload_packed.restype = C.c_int
    lib.lgr_stream.argtypes = [C.c_void_p]
    lib.lgr_stream.restype = C.c_void_p
    lib.lgr_format_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.lgr_format_create.restype = C.c_int
    lib.lgr_format_destroy.argtypes = [C.c_void_p]
    lib.lgr_format_destroy.restype = None
    lib.lgr_format_last_error.argtypes = [C.c_void_p]
    lib.lgr_format_last_error.restype = C.c_char_p
    lib.lgr_format_metrics.argtypes = [C.c_void_p, C.POINTER(LgrEvidenceIn), C.c_void_p, C.POINTER(C.c_float)]
    lib.lgr_format_metrics.restype = C.c_int
    lib.lgr_format_from_assign.argtypes = [C.c_void_p, C.POINTER(LgrAssignBatch), C.c_void_p, C.c_int32, C.c_void_p,
                                           C.POINTER(C.c_int32), C.POINTER(C.c_float)]
    lib.lgr_format_from_assign.restype = C.c_int
    lib.lgr_resident_assign.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]
    lib.lgr_resident_assign.restype = C.c_int
    lib.lgr_format_debug_evidence.argtypes = [C.c_void_p, C.POINTER(LgrEvidenceIn)]
    lib.lgr_format_debug_evidence.restype = C.c_int
    lib.lgr_format_packed_bytes.argtypes = [C.POINTER(LgrEvidenceIn)]
    lib.lgr_format_packed_bytes.restype = C.c_size_t
    lib.lgr_format_pack.argtypes = [C.POINTER(LgrEvidenceIn), C.c_void_p, C.c_size_t, C.POINTER(LgrFmtDir)]
    lib.lgr_format_pack.restype = C.c_int
    lib.lgr_format_metrics_packed.argtypes = [C.c_void_p, C.POINTER(LgrFmtPackedIn), C.c_void_p, C.POINTER(C.c_float)]
    lib.lgr_format_metrics_packed.restype = C.c_int
    lib.lgr_format_reserve.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int64]
    lib.lgr_format_reserve.restype = C.c_int
    lib.lgr_format_device_bytes.argtypes = [C.c_void_p]
    lib.lgr_format_device_bytes.restype = C.c_int64
    lib.lgr_repeat_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.lgr_repeat_create.restype = C.c_int
    lib.lgr_repeat_destroy.argtypes = [C.c_void_p]
    lib.lgr_repeat_destroy.restype = None
    lib.lgr_repeat_last_error.argtypes = [C.c_void_p]
    lib.lgr_repeat_last_error.restype = C.c_char_p
    lib.lgr_repeat_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.POINTER(C.c_float)]
    lib.lgr_repeat_scan.restype = C.c_int
    lib.lgr_repeat_reserve.argtypes = [C.c_void_p, C.c_int64, C.c_int32]
    lib.lgr_repeat_reserve.restype = C.c_int
    return lib
