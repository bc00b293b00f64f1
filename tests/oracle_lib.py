"""Loader for the CPU oracle (TEST INFRASTRUCTURE: oracle/liblancet_oracle.so)."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from lancet2_b200 import abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liblancet_oracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "liblancet_ref_scoring.so")

NATIVE_FLAGS = "-O3 -march=native -std=c++17 -fPIC -ffp-contract=off -pthread"
PORTABLE_FLAGS = "-O2 -std=c++17 -fPIC -ffp-contract=off -pthread"

_lib = None
_native = None


def build_oracle():
    subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, "liblancet_oracle.so"])


def load_native_oracle():
    """The oracle compiled ON THIS HOST with -O3 -march=native (SURVEY.md §8d asks for that build as the
    CPU baseline).  build() makes the portable -O2 library; a -march=native binary cannot travel to
    another machine's CPU, so it is compiled where it runs, into a temporary directory that is removed
    once the library is loaded (the repository tree may be read-only).  Returns (lib, flags); falls back
    to the portable build."""
    global _native
    if _native is not None:
        return _native
    try:
        srcs = [os.path.join(ORACLE_DIR, f) for f in ("mm2_restate.cpp", "genotype_oracle.cpp")]
        with tempfile.TemporaryDirectory(prefix="lancet2_b200_oracle_") as tmp:
            so = os.path.join(tmp, "liblancet_oracle_native.so")
            subprocess.check_call(["g++"] + NATIVE_FLAGS.split() + ["-shared", "-o", so] + srcs,
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            _native = (_bind(C.CDLL(so)), NATIVE_FLAGS)
    except Exception:  # noqa: BLE001 — no compiler on the box: the portable build is still a valid baseline
        _native = (load_oracle(), PORTABLE_FLAGS)
    return _native


def load_oracle() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(ORACLE_SO):
        build_oracle()
    _lib = _bind(C.CDLL(ORACLE_SO))
    return _lib


def _bind(lib):
    lib.orc_genotype_batch.argtypes = [C.POINTER(abi.LgrParams), C.POINTER(abi.LgrBatchIn),
                                       C.POINTER(abi.LgrBatchOut), C.c_int, C.POINTER(abi.LgrStats)]
    lib.orc_genotype_batch.restype = C.c_int
    lib.orc_default_params.argtypes = [C.POINTER(abi.LgrParams)]
    lib.orc_default_params.restype = None
    lib.orc_sketch.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.orc_sketch.restype = C.c_int
    lib.orc_hap_mid_occ.argtypes = [C.POINTER(abi.LgrParams), C.c_char_p, C.c_int]
    lib.orc_hap_mid_occ.restype = C.c_int
    lib.orc_map_debug.argtypes = [C.POINTER(abi.LgrParams), C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_uint32,
                                  C.c_int32, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int, C.POINTER(C.c_int32), C.c_void_p, C.c_int,
                                  C.POINTER(C.c_int32)]
    lib.orc_map_debug.restype = C.c_int
    lib.orc_extz.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                             C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    lib.orc_extz.restype = C.c_int
    lib.orc_edit_distance.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    lib.orc_edit_distance.restype = C.c_uint32
    lib.orc_refpos_to_qpos.argtypes = [C.c_void_p, C.c_int, C.c_uint64]
    lib.orc_refpos_to_qpos.restype = C.c_uint64
    lib.orc_softclip_penalty.argtypes = [C.c_void_p, C.c_int]
    lib.orc_softclip_penalty.restype = C.c_double
    lib.orc_local_score.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                    C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.orc_local_score.restype = None
    lib.orc_phred_err.argtypes = [C.c_uint32]
    lib.orc_phred_err.restype = C.c_double
    lib.orc_lancet_encode.argtypes = [C.c_uint8]
    lib.orc_lancet_encode.restype = C.c_uint8
    lib.orc_x31_hash.argtypes = [C.c_char_p]
    lib.orc_x31_hash.restype = C.c_uint32
    return lib


def default_params() -> abi.LgrParams:
    p = abi.LgrParams()
    load_oracle().orc_default_params(C.byref(p))
    return p


def oracle_genotype(batch: abi.Batch, params: abi.LgrParams = None, n_threads: int = 1, arena: int = 1 << 20, lib=None):
    lib = lib or load_oracle()
    params = params or default_params()
    res = abi.Result(batch, arena)
    bi, bo = batch.c_struct(), res.c_struct()
    st = abi.LgrStats()
    rc = lib.orc_genotype_batch(C.byref(params), C.byref(bi), C.byref(bo), n_threads, C.byref(st))
    if rc != 0:
        raise RuntimeError(f"oracle rc={rc}")
    return res, st


def map_debug(hap: bytes, read: bytes, name: str = "r0", params=None, mid_occ: int = 0, cap: int = 4096):
    lib = load_oracle()
    params = params or default_params()
    aln = np.zeros(1, dtype=abi.ALN_DTYPE)
    cig = np.zeros(cap, dtype=np.uint32)
    ax = np.zeros(cap, dtype=np.uint64)
    ay = np.zeros(cap, dtype=np.uint64)
    f = np.zeros(cap, dtype=np.int32)
    p = np.zeros(cap, dtype=np.int32)
    u = np.zeros(cap, dtype=np.uint64)
    na, nu = C.c_int32(0), C.c_int32(0)
    n = lib.orc_map_debug(C.byref(params), hap, len(hap), read, len(read), abi.x31_hash(name), mid_occ,
                          aln.ctypes.data, cig.ctypes.data, cap, ax.ctypes.data, ay.ctypes.data, f.ctypes.data,
                          p.ctypes.data, cap, C.byref(na), u.ctypes.data, cap, C.byref(nu))
    a = aln[0]
    return dict(n_regs=n, aln=a, cigar=[int(c) for c in cig[:int(a["n_cigar"])]],
                cigar_str="".join(f"{int(c) >> 4}{'MIDNSHP=XB'[int(c) & 0xf]}" for c in cig[:int(a["n_cigar"])]),
                anchors=list(zip(ax[:na.value].tolist(), ay[:na.value].tolist())), f=f[:na.value].tolist(),
                p=p[:na.value].tolist(), u=u[:nu.value].tolist())
