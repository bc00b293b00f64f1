"""The FORMAT row in Lancet2's per-window call pattern: lgr_format_metrics_packed (windows packed once, one copy per
batch, k_fmt_unpack) and lancet_gpu::FormatCalculator (many threads, one window per blocking call).  Every record must
equal lgr_format_metrics on the same supports byte for byte: a support's result does not depend on its batch."""
import ctypes as C

import numpy as np
import pytest

import format_lib as F
from lancet2_b200 import abi
from lancet2_b200.format_metrics import FormatCalculator, GpuFormatMetrics, PackedWindows, private_contexts_run

pytestmark = pytest.mark.gpu
LGR_E_ARG = -1


@pytest.fixture(scope="module")
def fmt():
    f = GpuFormatMetrics(0)
    yield f
    f.close()


def cut(sups, rng, max_len=8, empty_frac=0.1):
    """sups cut into consecutive windows of random size, some of them empty"""
    wins, i = [], 0
    while i < len(sups):
        if rng.random() < empty_frac:
            wins.append([])
            continue
        n = int(rng.integers(1, max_len + 1))
        wins.append(sups[i:i + n])
        i += n
    return wins


def same_bytes(fmt, windows, **kw):
    """packed records of the windows == lgr_format_metrics on all their supports; returns the records"""
    flat = [s for w in windows for s in w]
    want, _ = fmt.compute(flat)
    rc_plain = fmt.last_rc
    got, ms = fmt.compute_packed(windows, **kw)
    assert fmt.last_rc == rc_plain
    assert got.tobytes() == want.tobytes()
    return got, ms


def random_windows(seed, n_sup=3000, max_len=8):
    rng = np.random.default_rng(seed)
    sups = [F.random_support(rng, n=0 if rng.random() < 0.05 else None) for _ in range(n_sup)]
    return cut(sups, rng, max_len)


def test_packed_golden_supports(fmt):
    sups, want, _ = F.load_golden()
    got, ms = same_bytes(fmt, cut(sups, np.random.default_rng(1)))
    errs = F.compare_format(want, got)
    assert not errs, "\n".join(errs[:20])
    assert ms > 0.0


def test_packed_edge_supports(fmt):
    sups, want = F.load_golden_edge()
    got, _ = same_bytes(fmt, cut(sups, np.random.default_rng(2), max_len=4))
    errs = F.compare_format(want, got)
    assert not errs, "\n".join(errs[:20])
    same_bytes(fmt, [F.edge_supports()])


def test_packed_random_windows_equal_each_window_alone(fmt):
    wins = random_windows(3)
    got, _ = same_bytes(fmt, wins)
    starts = np.concatenate([[0], np.cumsum([len(w) for w in wins])])
    for i in range(0, len(wins), 17):  # a window alone through both paths, against its slice of the batch
        w, at = wins[i], int(starts[i])
        if not w:
            continue
        alone, _ = fmt.compute(w)
        assert alone.tobytes() == got[at:at + len(w)].tobytes()
        assert fmt.compute_packed([w])[0].tobytes() == alone.tobytes()


def test_packed_wide_supports(fmt):
    rng = np.random.default_rng(4)
    sups = [F.random_support(rng, n_alleles=int(rng.choice([2, 3, 8, 9, 12]))) for _ in range(400)]
    got, _ = same_bytes(fmt, cut(sups, rng))
    assert fmt.last_rc == abi.LGR_E_PARTIAL
    wide = got["n_alleles"] > abi.LGR_FMT_MAX_ALLELES
    assert wide.any() and (got["valid"][wide] == abi.LGR_FMT_WIDE).all()


def test_packed_more_supports_than_resident_ctas(fmt):
    rng = np.random.default_rng(5)
    sups = [F.random_support(rng, n=int(rng.integers(0, 24))) for _ in range(6000)]
    same_bytes(fmt, cut(sups, rng, max_len=40))


def test_packed_directory_outside_the_slab(fmt):
    same_bytes(fmt, random_windows(6, n_sup=500), dir_inside=False)


def test_packed_one_window_larger_than_the_rest(fmt):
    rng = np.random.default_rng(7)
    big = [F.random_support(rng, n=int(rng.integers(200, 1200))) for _ in range(60)]
    small = [[F.random_support(rng, n=5)] for _ in range(20)]
    same_bytes(fmt, small[:10] + [big] + small[10:])


def _call(fmt, pk):
    out = np.zeros(max(pk.n_supports, 1), dtype=abi.FORMAT_DTYPE)
    st = pk.c_struct()
    return fmt._main.lgr_format_metrics_packed(fmt._ctx, C.byref(st), out.ctypes.data, None)


def test_bad_directories_are_refused_and_the_next_call_succeeds(fmt):
    wins = random_windows(8, n_sup=60)
    want, _ = fmt.compute([s for w in wins for s in w])

    def magic(pk):
        pk.slab[int(pk.dir[1]["rec_off"])] ^= 0xFF

    def bases(pk):
        pk.dir[2]["sup_base"] += 1

    def ev_bases(pk):
        pk.dir[3]["ev_base"] -= 1

    def rec_off(pk):
        pk.dir[2]["rec_off"] = pk.slab_bytes + 16

    def rec_off_unaligned(pk):
        pk.dir[1]["rec_off"] += 8

    def counts(pk):
        pk.dir[1]["n_evidence"] += 1

    for bad in (magic, bases, ev_bases, rec_off, rec_off_unaligned, counts):
        pk = PackedWindows(wins, fmt._main)
        bad(pk)
        assert _call(fmt, pk) == LGR_E_ARG, bad.__name__
        got, _ = fmt.compute_packed(wins)
        assert got.tobytes() == want.tobytes()


def test_malformed_records_in_the_slab_are_refused(fmt):
    # the host never reads the records: the device finds an allele >= K or a broken sup_begin and computes nothing wrong
    rng = np.random.default_rng(9)
    wins = [[F.random_support(rng, n=20, n_alleles=2) for _ in range(3)] for _ in range(4)]
    want, _ = fmt.compute([s for w in wins for s in w])
    hdr = 160
    for what in ("allele", "sup_begin"):
        pk = PackedWindows(wins, fmt._main)
        base = int(pk.dir[2]["rec_off"])
        S, N = 3, 60
        if what == "allele":
            off = hdr + 16 * 2 + 4 * ((N * 8 + 15) // 16 * 16) + 3 * 16 + 4 * ((N * 4 + 15) // 16 * 16)
            pk.slab[base + off + 5] = 7
        else:
            pk.slab[base + hdr + 8:base + hdr + 16] = np.frombuffer(np.int64(1 << 40).tobytes(), np.uint8)
        assert _call(fmt, pk) == LGR_E_ARG, what
        got, _ = fmt.compute_packed(wins)
        assert got.tobytes() == want.tobytes()


def test_reserve_keeps_device_bytes(fmt):
    f = GpuFormatMetrics(0)
    try:
        wins = random_windows(10, n_sup=800)
        pk = PackedWindows(wins, f._main)
        f.reserve(pk.slab_bytes, pk.n_supports, pk.n_evidence)
        held = f.device_bytes()
        for w in (wins, wins[: len(wins) // 2], wins[::3]):
            same_bytes(f, w)
            assert f.device_bytes() == held
        big = random_windows(11, n_sup=3000)
        same_bytes(f, big)
        assert f.device_bytes() > held
    finally:
        f.close()


def _alone(fmt, wins):
    out = []
    for w in wins:
        out.append(fmt.compute(w)[0] if w else np.zeros(0, abi.FORMAT_DTYPE))
    return out


@pytest.mark.parametrize("threads", [1, 8, 32])
def test_calculator_threads(fmt, threads):
    wins = random_windows(20 + threads, n_sup=1500, max_len=6)
    want = _alone(fmt, wins)
    calc = FormatCalculator(0)
    try:
        got, status, ctr = calc.run(wins, threads=threads)
    finally:
        calc.close()
    assert (status == 0).all()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(want, got))
    assert ctr["windows"] == sum(1 for w in wins if w) and ctr["alone"] == 0
    assert ctr["supports"] == sum(len(w) for w in wins)
    if threads == 32:
        assert ctr["max_windows_in_batch"] > 1
    priv, pstatus, _ = private_contexts_run(wins, threads=threads)
    assert (pstatus == 0).all() and all(a.tobytes() == b.tobytes() for a, b in zip(want, priv))


def test_calculator_failure_isolation(fmt):
    rng = np.random.default_rng(30)
    wins = random_windows(31, n_sup=600, max_len=5)
    bad = [F.random_support(rng, n=10, n_alleles=2)]
    bad[0]["allele"] = np.full(10, 2)  # allele >= K
    wins.insert(17, bad)
    want = _alone(fmt, [w if i != 17 else [] for i, w in enumerate(wins)])
    calc = FormatCalculator(0)
    try:
        got, status, _ = calc.run(wins, threads=16)
    finally:
        calc.close()
    assert status[17] == 1 and (np.delete(status, 17) == 0).all()
    assert all(a.tobytes() == b.tobytes() for i, (a, b) in enumerate(zip(want, got)) if i != 17)


def test_calculator_oversized_window(fmt):
    rng = np.random.default_rng(40)
    big = [F.random_support(rng, n=400) for _ in range(20)]
    wins = [[F.random_support(rng, n=10)] for _ in range(30)]
    wins.insert(5, big)
    want = _alone(fmt, wins)
    calc = FormatCalculator(0, slab_bytes=64 << 10)
    try:
        got, status, ctr = calc.run(wins, threads=4)
    finally:
        calc.close()
    assert (status == 0).all() and ctr["alone"] == 1
    assert all(a.tobytes() == b.tobytes() for a, b in zip(want, got))


def test_calculator_end_to_end_from_a_realignment_batch():
    from test_zz_format_adapter import call_args, make_case, python_model
    lib = abi.load_library()
    groups, batch, names, meta, want = make_case()
    sups, keys = python_model(groups, batch, names, meta, want)
    lib.lgr_adapter_format_calculator_columns.argtypes = [C.c_int, C.POINTER(abi.LgrBatchIn), C.c_char_p, C.c_char_p] + \
        [C.c_void_p] * 7 + [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_char_p, C.c_int]
    lib.lgr_adapter_format_calculator_columns.restype = C.c_int
    calc_out = np.zeros(len(keys), dtype=abi.FORMAT_DTYPE)
    plain_out = np.zeros(len(keys), dtype=abi.FORMAT_DTYPE)
    err = C.create_string_buffer(512)
    args, _bi = call_args(batch, names, meta, want)
    n = lib.lgr_adapter_format_calculator_columns(0, *args, 4, calc_out.ctypes.data, plain_out.ctypes.data, len(keys), err, len(err))
    assert n == len(keys), err.value.decode()
    assert calc_out.tobytes() == plain_out.tobytes()
    rc, emu = F.emu_format(sups)
    assert rc == 0
    errs = F.compare_format(emu, calc_out)
    assert not errs, "\n".join(errs[:20])
