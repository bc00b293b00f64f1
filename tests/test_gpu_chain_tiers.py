"""The chain stage runs in two tiers: k_chain_lean takes every pair and finishes the sorted co-linear
ones; every other shape is queued for k_chain_cold.  One small group per shape, each checked against
the CPU oracle and against the device counters that say where its pairs went."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
from compare import compare_results
from lancet2_b200 import abi, synth

pytestmark = pytest.mark.gpu

# indices into the device counters (enum Ctr in lancet2_b200/csrc/lgr_dev.cuh; names in tools/debug_counters.py)
NCOLD, COLD_SORT, LEAN_DEFER = 24, 27, 29
_COMP = bytes.maketrans(b"ACGT", b"TGCA")


def _group(ref, alt, starts, src, rng):
    """haplotypes [ref, alt], one variant over both, and one error-free forward read of 150 bp per start,
    cut from haplotype `src`"""
    haps = [ref, alt]
    reads = [haps[src][s:s + 150].tobytes() for s in starts]
    quals = [bytes(rng.integers(20, 41, 150, dtype=np.uint8)) for _ in starts]
    names = [f"t{i}" for i in range(len(starts))]
    variants = [[(300, 1, 0), (300, 1, 1)]]
    return abi.Group(haps=[h.tobytes() for h in haps], reads=reads, quals=quals, names=names, variants=variants)


def _snv(ref, pos):
    alt = ref.copy()
    alt[pos] = b"C"[0] if ref[pos] != b"C"[0] else b"G"[0]
    return alt


def clean():
    rng = np.random.default_rng(101)
    ref = synth._rand_bases(rng, 800)
    return _group(ref, _snv(ref, 300), [400, 450, 500], 0, rng)


def deletion():
    # the reads come from the haplotype with a 5 bp deletion and span it: co-linear against that
    # haplotype, two diagonals against the other one
    rng = np.random.default_rng(102)
    ref = synth._rand_bases(rng, 800)
    alt = np.concatenate([ref[:400], ref[405:]])
    return _group(ref, alt, [330, 340, 350], 1, rng)


def palindrome():
    # an inverted repeat: the reverse complement of ref[200:240] also sits at 600:640, so the reads'
    # minimizers there hit the reverse strand too and their anchor list is not sorted
    rng = np.random.default_rng(103)
    ref = synth._rand_bases(rng, 800)
    ref[600:640] = np.frombuffer(ref[200:240].tobytes().translate(_COMP)[::-1], dtype=np.uint8)
    return _group(ref, _snv(ref, 300), [150, 160, 170], 0, rng)


def tandem():
    # the other haplotype carries a 60 bp dinucleotide repeat, and so do the reads: its minimizers occur
    # there more often than mid_occ, which the repeat-free first haplotype sets
    rng = np.random.default_rng(104)
    left, right = synth._rand_bases(rng, 380), synth._rand_bases(rng, 380)
    alt = np.concatenate([left, np.tile(np.frombuffer(b"AC", dtype=np.uint8), 30), right])
    return _group(np.concatenate([left, right]), alt, [340, 350, 360], 1, rng)


@pytest.fixture(scope="module")
def gpu():
    from lancet2_b200.realign import GpuRealigner
    g = GpuRealigner(0)
    g.lib.lgr_debug_counters.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    g.lib.lgr_debug_counters.restype = C.c_int
    yield g
    g.close()


@pytest.mark.parametrize("make,deferred,unsorted", [(clean, False, False), (deletion, True, False),
                                                    (palindrome, True, True), (tandem, True, None)])
def test_chain_tier_matches_oracle(gpu, make, deferred, unsorted):
    batch = abi.Batch([make()])
    want, st = O.oracle_genotype(batch, gpu.params)
    got, st2 = gpu.genotype_batch(batch)
    errs = compare_results(batch, want, got)
    assert not errs, "\n".join(errs[:20])
    # every pair counted once, where it completes
    assert (st.chain_evals, st.n_anchors, st.dp_cells_full, st.n_aligned) == \
        (st2.chain_evals, st2.n_anchors, st2.dp_cells_full, st2.n_aligned)
    buf = (C.c_longlong * 64)()
    n = gpu.lib.lgr_debug_counters(gpu._ctx, buf, 64)
    ctr = [int(buf[i]) for i in range(n)]
    where = f"NCOLD={ctr[NCOLD]} COLD_SORT={ctr[COLD_SORT]} LEAN_DEFER={ctr[LEAN_DEFER]}"
    assert (ctr[LEAN_DEFER] > 0) == deferred, where
    assert ctr[NCOLD] >= ctr[LEAN_DEFER], where
    if unsorted is not None:
        assert (ctr[COLD_SORT] > 0) == unsorted, where
