"""The packed evidence wire format of the FORMAT row (lgr_format_packed_bytes / lgr_format_pack), on the host only:
an independent numpy decoder reads every block back, and every input lgr_format_metrics refuses is refused here too."""
import ctypes as C

import numpy as np
import pytest

import format_lib as F
from lancet2_b200 import abi

LGR_E_ARG = -1


@pytest.fixture(scope="module")
def lib():
    import os
    if not os.path.exists(abi.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return abi.load_library()


def up16(x):
    return (x + 15) & ~15


def decode_block(buf: bytes):
    """header + sections of one block, from the bytes alone (the layout restated, not taken from the library)"""
    hdr = np.frombuffer(buf[:160], dtype=np.dtype([("magic", "<u4"), ("S", "<i4"), ("N", "<i8"), ("rec_bytes", "<u8"),
                                                   ("reserved", "<u8"), ("off", "<u8", (16,))]))[0]
    S, N = int(hdr["S"]), int(hdr["N"])
    off, o = [], 160
    for _, dt, kind in abi.FMT_SECTIONS:
        n = S + 1 if kind == "S+1" else S if kind == "S" else N
        off.append(o)
        o += up16(n * np.dtype(dt).itemsize)
    assert [int(x) for x in hdr["off"]] == off
    assert int(hdr["rec_bytes"]) == o and o % 16 == 0
    cols = {}
    for (name, dt, kind), at in zip(abi.FMT_SECTIONS, off):
        n = S + 1 if kind == "S+1" else S if kind == "S" else N
        nbytes = n * np.dtype(dt).itemsize
        cols[name] = np.frombuffer(buf[at:at + nbytes], dtype=dt)
        assert not any(buf[at + nbytes:at + up16(nbytes)]), f"{name}: padding not zero"
    return int(hdr["magic"]), S, N, o, cols


def pack(lib, sups, cap=None):
    batch = abi.EvidenceBatch(sups)
    st = batch.c_struct()
    need = int(lib.lgr_format_packed_bytes(C.byref(st)))
    buf = np.full((cap if cap is not None else need) + 16, 0xAB, dtype=np.uint8)
    d = abi.LgrFmtDir()
    rc = lib.lgr_format_pack(C.byref(st), buf.ctypes.data, cap if cap is not None else need, C.byref(d))
    return rc, need, buf, d, batch


def check_round_trip(lib, sups):
    rc, need, buf, d, batch = pack(lib, sups)
    assert rc == 0
    assert need % 16 == 0 and need > 0
    magic, S, N, used, cols = decode_block(buf.tobytes())
    assert magic == abi.LGR_FMT_MAGIC and (S, N) == (batch.n_supports, batch.n_evidence) and used <= need
    assert (d.n_supports, d.n_evidence, d.rec_off, d.sup_base, d.ev_base) == (S, N, 0, 0, 0)
    assert d.n_wide == int((batch.sup_n_alleles > abi.LGR_FMT_MAX_ALLELES).sum())
    for name in ("sup_begin", "sup_n_alleles", "sup_variant_len", "sup_total_haps"):
        assert np.array_equal(cols[name], getattr(batch, name)), name
    for name, _ in abi.EVIDENCE_FIELDS:
        assert np.array_equal(cols[name], batch.cols[name]), name
    assert all(buf[need:need + 16] == 0xAB)  # nothing written past the size it announced


def test_round_trip_random_windows(lib):
    rng = np.random.default_rng(7)
    for _ in range(60):
        n_sup = int(rng.integers(1, 9))
        sups = []
        for _ in range(n_sup):
            k = int(rng.choice([1, 2, 3, 8, 9, 12]))
            sups.append(F.random_support(rng, n=int(rng.integers(0, 40)), n_alleles=k))
        check_round_trip(lib, sups)


@pytest.mark.parametrize("n", list(range(1, 18)))
def test_round_trip_alignment_edges(lib, n):
    rng = np.random.default_rng(100 + n)
    check_round_trip(lib, [F.random_support(rng, n=n, n_alleles=2)])
    check_round_trip(lib, [F.random_support(rng, n=0), F.random_support(rng, n=n, n_alleles=1),
                           F.random_support(rng, n=0, n_alleles=3)])


def test_window_without_supports_or_records(lib):
    rc, need, buf, d, _ = pack(lib, [])
    assert rc == 0 and (d.n_supports, d.n_evidence) == (0, 0)
    magic, S, N, used, cols = decode_block(buf.tobytes())
    assert (magic, S, N) == (abi.LGR_FMT_MAGIC, 0, 0) and used == need and list(cols["sup_begin"]) == [0]
    rng = np.random.default_rng(3)
    check_round_trip(lib, [F.random_support(rng, n=0) for _ in range(5)])  # supports, N = 0


def test_packed_bytes_is_an_upper_bound_multiple_of_16(lib):
    rng = np.random.default_rng(11)
    for _ in range(40):
        sups = [F.random_support(rng, n=int(rng.integers(0, 30))) for _ in range(int(rng.integers(0, 6)))]
        rc, need, buf, _, _ = pack(lib, sups)
        assert rc == 0 and need % 16 == 0
        assert decode_block(buf.tobytes())[3] <= need


def _malformed(lib, sups, mutate):
    batch = abi.EvidenceBatch(sups)
    st = batch.c_struct()
    need = int(lib.lgr_format_packed_bytes(C.byref(st)))
    mutate(batch, st)
    buf = np.zeros(max(need, 1 << 16), dtype=np.uint8)
    return lib.lgr_format_pack(C.byref(st), buf.ctypes.data, len(buf), None)


def test_malformed_windows_are_refused(lib):
    rng = np.random.default_rng(5)
    sups = [F.random_support(rng, n=6, n_alleles=2), F.random_support(rng, n=5, n_alleles=3)]
    ok = _malformed(lib, sups, lambda b, st: None)
    assert ok == 0

    def neg_s(b, st):
        st.n_supports = -1

    def neg_n(b, st):
        st.n_evidence = -1

    def begin0(b, st):
        b.sup_begin[0] = 1

    def begin_end(b, st):
        b.sup_begin[-1] = b.n_evidence + 1

    def not_monotone(b, st):
        b.sup_begin[1] = b.n_evidence + 1  # ends still [0, N], the middle past the end

    def zero_k(b, st):
        b.sup_n_alleles[1] = 0

    def missing_sup(b, st):
        st.sup_total_haps = None

    def missing_col(b, st):
        st.hap_id = None

    def allele_ge_k(b, st):
        b.cols["allele"][7] = 3  # support 1 has K = 3

    for mutate in (neg_s, neg_n, begin0, begin_end, not_monotone, zero_k, missing_sup, missing_col, allele_ge_k):
        assert _malformed(lib, sups, mutate) == LGR_E_ARG, mutate.__name__
    assert lib.lgr_format_pack(None, None, 0, None) == LGR_E_ARG


def test_packed_bytes_zero_for_malformed(lib):
    st = abi.LgrEvidenceIn()
    st.n_supports = -1
    assert lib.lgr_format_packed_bytes(C.byref(st)) == 0
    st.n_supports, st.n_evidence = 1, -5
    assert lib.lgr_format_packed_bytes(C.byref(st)) == 0
    assert lib.lgr_format_packed_bytes(None) == 0


def test_small_cap_is_refused(lib):
    rng = np.random.default_rng(9)
    sups = [F.random_support(rng, n=13, n_alleles=2)]
    _, need, _, _, _ = pack(lib, sups)
    rc, _, buf, _, _ = pack(lib, sups, cap=need - 16)
    assert rc == LGR_E_ARG
    assert all(buf == 0xAB)  # nothing written


def test_new_symbols_are_exported(lib):
    for sym in ("lgr_format_packed_bytes", "lgr_format_pack", "lgr_format_metrics_packed", "lgr_format_reserve",
                "lgr_format_device_bytes", "lgr_adapter_format_calculator_create", "lgr_adapter_format_calculator_run",
                "lgr_adapter_format_calculator_destroy", "lgr_adapter_format_private_run",
                "lgr_adapter_format_calculator_columns"):
        assert hasattr(lib, sym), sym
    assert {"lgr_format_packed_bytes", "lgr_format_pack", "lgr_format_metrics_packed", "lgr_format_reserve",
            "lgr_format_device_bytes"} <= set(abi.declared_symbols())
    assert C.sizeof(abi.LgrFmtDir) == 48 and C.sizeof(abi.LgrFmtBlkHdr) == 160
