"""The repeat check in Lancet2's call pattern: k_repeat_scan's diagonal slices (small batches spread over the GPU) and
lancet_gpu::RepeatChecker (many threads, one window per blocking call), every answer bit-equal to the CPU oracle."""
import numpy as np
import pytest

import repeat_lib
from lancet2_b200 import abi
from lancet2_b200.repeat_scan import ONE_SLICE_LIBRARY, GpuRepeatScan, RepeatChecker

ORC = repeat_lib.oracle()
K_LOOP = tuple(range(13, 128, 6))  # Lancet2's defaults: min_k 13, max_k 127, step 6
WARPS = 8                           # warps of k_repeat_scan's CTA: a slice takes 8 consecutive diagonals per round


def _expect(seq, questions):
    return np.array([ORC.orc_has_repeat(seq, len(seq), k, mm) for k, mm in questions], dtype=np.uint8)


def _resident():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * 8


def _plant_on_diagonal(seq, k, d, at=0):
    """the k-mer at `at + d` becomes a copy of the one at `at` (left to right, so a short d gives a period-d run)"""
    s = bytearray(seq)
    for p in range(k):
        s[at + d + p] = s[at + p]
    return bytes(s)


def _slice_ends(S, d_max):
    """first and last diagonal of every slice s of S (slice s takes 1 + s * 8 + warp, stepping by S * 8)"""
    out = []
    for s in range(S):
        mine = [d for d in range(1 + s * WARPS, d_max + 1) if (d - 1) % (S * WARPS) // WARPS == s]
        if mine:
            out += [mine[0], mine[-1]]
    return out


def _scan_both(jobs):
    """answers of the shipped build and of the one-slice build (every group on one CTA), which must agree"""
    got, _ = GpuRepeatScan().scan(jobs)
    one, _ = GpuRepeatScan(library=ONE_SLICE_LIBRARY).scan(jobs)
    assert np.array_equal(got, one)
    return got


def _oracle_jobs(jobs):
    return np.array([ORC.orc_has_repeat(s, len(s), k, mm) for s, k, mm in jobs], dtype=np.uint8)


@pytest.fixture(scope="module")
def lib():
    import os
    if not os.path.exists(abi.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return abi.load_library()


def test_checker_without_gpu_fails_loudly(lib):
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("a GPU is present")
    except ImportError:
        pass
    with pytest.raises(RuntimeError):
        RepeatChecker()


# ---- the slice schedule of k_repeat_scan ----

@pytest.mark.gpu
@pytest.mark.parametrize("S", [2, 3, 7, "max"])
def test_repeats_on_first_and_last_diagonal_of_every_slice(S):
    rng = np.random.default_rng(7)
    k, mm, n = 40, 2, 300
    resident = _resident()
    if S == "max":
        # one window alone: as many slices as its diagonals allow (8 per slice)
        S = (n - k) // WARPS
        targets = _slice_ends(S, n - k)
        for d in targets:
            seq = _plant_on_diagonal(repeat_lib.random_window(rng, n), k, d, at=int(rng.integers(0, n - k - d + 1)))
            jobs = [(seq, k, mm)]
            got = _scan_both(jobs)
            assert got.tolist() == _oracle_jobs(jobs).tolist() == [1], d
        return
    n_windows = resident // S
    assert resident // n_windows == S  # the batch size that gives exactly S slices per group
    targets = _slice_ends(S, n - k)
    jobs = []
    for w in range(n_windows):
        seq = repeat_lib.random_window(rng, n)
        if w % 3:  # a third of the windows carry no planted repeat
            d = targets[w % len(targets)]
            seq = _plant_on_diagonal(seq, k, d, at=int(rng.integers(0, n - k - d + 1)))
        jobs.append((seq, k, mm))
    got = _scan_both(jobs)
    want = _oracle_jobs(jobs)
    assert np.array_equal(got, want)
    assert want.sum() >= 2 * n_windows // 3


@pytest.mark.gpu
def test_first_and_last_diagonal_of_a_lone_window():
    rng = np.random.default_rng(8)
    for n, k in ((1000, 31), (2500, 61)):
        for d in (1, n - k):
            seq = _plant_on_diagonal(repeat_lib.random_window(rng, n), k, d, at=0 if d > 1 else n // 2)
            jobs = [(seq, kk, 2) for kk in K_LOOP] + [(seq, max(K_LOOP), 0)]
            got = _scan_both(jobs)
            assert np.array_equal(got, _oracle_jobs(jobs))
            assert got[K_LOOP.index(k)] == 1


@pytest.mark.gpu
def test_only_the_smallest_k_hits_and_no_k_hits():
    rng = np.random.default_rng(9)
    base = repeat_lib.random_window(rng, 1500)
    small = bytearray(base)
    small[900:913] = small[100:113]  # one exact 13-mer repeat and nothing longer
    small = bytes(small)
    for seq, want_first in ((small, 1), (base, 0)):
        jobs = [(seq, k, 0) for k in K_LOOP]
        got = _scan_both(jobs)
        assert np.array_equal(got, _oracle_jobs(jobs))
        assert got.tolist() == [want_first] + [0] * (len(K_LOOP) - 1)


@pytest.mark.gpu
@pytest.mark.parametrize("mm", range(6))
def test_lengths_and_mismatch_counts(mm):
    rng = np.random.default_rng(100 + mm)
    k = 40
    jobs = []
    for n in (1, k, k + 1, 2500, abi.LGR_REPEAT_MAX_LEN):
        seq = repeat_lib.random_window(rng, n)
        if n > 2 * k:
            seq = repeat_lib.plant_repeat(rng, seq, k, 3, gap=n - k)  # 3 substitutions, on the last diagonal
        for kk in (k, 13):
            jobs.append((seq, kk, mm))
    for j in jobs:  # alone (all slices on one window) and together
        assert np.array_equal(_scan_both([j]), _oracle_jobs([j]))
    got = _scan_both(jobs)
    assert np.array_equal(got, _oracle_jobs(jobs))


def _windows(seed, n_windows, lengths=(200, 300, 400), k_values=(13, 19, 25, 31, 61)):
    jobs = repeat_lib.window_jobs(seed, n_windows, k_values=k_values, lengths=lengths)
    q = len(k_values) + 1
    return [(jobs[w * q][0], [(k, mm) for _, k, mm in jobs[w * q:(w + 1) * q]]) for w in range(n_windows)]


@pytest.mark.gpu
@pytest.mark.parametrize("size", [1, 2, 16, 17, "resident-1", "resident", "resident+1", 2000])
def test_both_schedules_agree_with_the_oracle(size):
    resident = _resident()
    n = {"resident-1": resident - 1, "resident": resident, "resident+1": resident + 1}.get(size, size)
    windows = _windows(30 + n, n)
    jobs = [(s, k, mm) for s, qs in windows for k, mm in qs]
    got = _scan_both(jobs)
    assert np.array_equal(got, _oracle_jobs(jobs))


@pytest.mark.gpu
def test_reserve_then_scan(lib):
    scan = GpuRepeatScan()
    assert lib.lgr_repeat_reserve(scan._ctx, 1 << 20, 4096) == 0
    assert lib.lgr_repeat_reserve(scan._ctx, -1, 4096) == -1
    jobs = repeat_lib.window_jobs(12, 20)
    got, _ = scan.scan(jobs)
    assert np.array_equal(got, _oracle_jobs(jobs))


# ---- lancet_gpu::RepeatChecker ----

@pytest.fixture(scope="module")
def checker_windows():
    """256 distinct windows of 300-600 bp, each asked Lancet2's k-loop with 2 mismatches and the exact question at max_k"""
    rng = np.random.default_rng(2026)
    windows, seen = [], set()
    while len(windows) < 256:
        n = int(rng.integers(300, 601))
        seq = repeat_lib.random_window(rng, n)
        kind = len(windows) % 4
        if kind == 1:
            seq = repeat_lib.plant_repeat(rng, seq, int(rng.choice(K_LOOP)), int(rng.integers(0, 4)))
        elif kind == 2:
            unit = repeat_lib.random_window(rng, int(rng.integers(1, 7)))
            seq = (seq[:50] + unit * 30 + seq[50:])[:n]
        if seq in seen:
            continue
        seen.add(seq)
        windows.append((seq, [(k, 2) for k in K_LOOP] + [(max(K_LOOP), 0)]))
    want = [_expect(s, q) for s, q in windows]
    return windows, want


@pytest.mark.gpu
@pytest.mark.parametrize("threads", [1, 4, 16, 64])
def test_checker_threads(checker_windows, threads):
    windows, want = checker_windows
    chk = RepeatChecker()
    got, status, ctr = chk.run(windows, threads=threads)
    chk.close()
    assert status.tolist() == [0] * len(windows)
    for w, (g, e) in enumerate(zip(got, want)):
        assert np.array_equal(g, e), w  # nothing lost or handed to another window
    assert ctr["windows"] == len(windows) and ctr["questions"] == sum(len(q) for _, q in windows)
    assert ctr["batches"] <= len(windows)
    if threads == 1:
        assert ctr["max_windows_in_batch"] == 1
    if threads == 16:
        assert ctr["max_windows_in_batch"] > 1


@pytest.mark.gpu
def test_destroying_the_checker_completes_its_waiting_callers(checker_windows):
    windows, want = checker_windows
    chk = RepeatChecker()
    got, status, _ = chk.run(windows[:64], threads=64, destroy=True)  # one window per thread
    assert status.tolist() == [0] * 64
    assert all(np.array_equal(g, e) for g, e in zip(got, want[:64]))
    with pytest.raises(RuntimeError):
        chk.run(windows[:1])


@pytest.mark.gpu
def test_too_long_window_and_bad_questions_stay_with_their_caller(checker_windows):
    windows, want = checker_windows
    rng = np.random.default_rng(4)
    too_long = (repeat_lib.random_window(rng, abi.LGR_REPEAT_MAX_LEN + 1), [(13, 2), (127, 0)])
    beyond = (repeat_lib.random_window(rng, 3 * abi.LGR_REPEAT_MAX_LEN), [(13, 2)])  # larger than the reserved batch
    bad_k = (windows[0][0], [(13, 2), (0, 2)])
    bad_mm = (windows[1][0], [(13, -1)])
    mixed = list(windows[2:40]) + [too_long, bad_k, beyond, bad_mm]
    chk = RepeatChecker(max_seq_bytes=2 * abi.LGR_REPEAT_MAX_LEN)
    got, status, ctr = chk.run(mixed, threads=16)
    chk.close()
    n = len(windows[2:40])
    assert status.tolist() == [0] * n + [0, 1, 0, 1]
    for g, e in zip(got[:n], want[2:40]):
        assert np.array_equal(g, e)
    assert got[n].tolist() == [abi.LGR_REPEAT_TOO_LONG] * 2
    assert got[n + 2].tolist() == [abi.LGR_REPEAT_TOO_LONG]
    assert ctr["windows"] == n + 1  # the 8,193-base window went through the device with its batch-mates
