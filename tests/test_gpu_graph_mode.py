"""Graph mode of the blocking calls (lgr_set_graph_mode): the device pass captured as one CUDA graph must give
exactly what the separate launches give, on every branch of the pass, reuse one executable per topology, keep the
overflow pass, the per-group status and the stage times, and work through the C++ adapter's direct path."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as O
from compare import compare_results
from lancet2_b200 import abi, synth


def _lib():
    if not os.path.exists(abi.LIB_PATH):
        import __graft_entry__ as ge
        ge.build()
    return abi.load_library()


def test_graph_mode_symbols_are_exported_and_declared():
    lib = _lib()
    for sym in ("lgr_set_graph_mode", "lgr_graph_counters"):
        assert sym in abi.declared_symbols() and hasattr(lib, sym)
    assert hasattr(lib, "lgr_adapter_direct_graph_run")
    # a NULL context is refused, not dereferenced
    n = C.c_int64(-1)
    assert lib.lgr_set_graph_mode(None, 1) == -1
    assert lib.lgr_graph_counters(None, C.byref(n), None, None) == -1 and n.value == -1


@pytest.fixture(scope="module")
def gpu():
    from lancet2_b200.realign import GpuRealigner
    g = GpuRealigner(0)
    yield g
    g.close()


def no_variants(groups):
    return [abi.Group(haps=g.haps, reads=g.reads, quals=g.quals, names=g.names, variants=[]) for g in groups]


def same_results(batch, a, b):
    """every aln field but the arena offset of a long CIGAR, every CIGAR, every assignment byte for byte"""
    errs = compare_results(batch, a, b)
    assert not errs, "\n".join(errs[:20])
    n = batch.n_pairs
    for f in abi.ALN_DTYPE.names:
        if f == "cigar_off":
            assert np.array_equal(a.aln[f][:n] < 0, b.aln[f][:n] < 0)
        else:
            assert np.array_equal(a.aln[f][:n], b.aln[f][:n]), f
    assert a.assign[:batch.n_assign].tobytes() == b.assign[:batch.n_assign].tobytes()
    assert np.array_equal(a.grp_mid_occ[:batch.n_groups], b.grp_mid_occ[:batch.n_groups])


def run_both(gpu, batch, packed=None):
    """the same batch with graph mode off, then on; (stream result, graph result, graph stats)"""
    def run():
        return gpu.genotype_packed(packed, batch) if packed is not None else gpu.genotype_batch(batch)
    gpu.set_graph_mode(False)
    ref, st0 = run()
    gpu.set_graph_mode(True)
    try:
        got, st1 = run()
    finally:
        gpu.set_graph_mode(False)
    assert (st0.n_pairs, st0.n_aligned, st0.chain_evals, st0.n_anchors, st0.dp_cells_full, st0.kernel_launches) == \
        (st1.n_pairs, st1.n_aligned, st1.chain_evals, st1.n_anchors, st1.dp_cells_full, st1.kernel_launches)
    return ref, got, st1


@pytest.mark.gpu
def test_every_branch_matches_stream_mode_and_oracle(gpu):
    """1 / 4 / 16 groups, reads of 150 and 250 bases (both chain workspace sizes), a batch without variants, each as
    the plain SoA input (k_encode) and as the packed input (unpack kernels), in one context"""
    l150 = synth.make_region_groups(21, ref_len=70_000)
    l250 = synth.make_region_groups(22, ref_len=8_000, read_len=250)
    cases = {"1g": l150[:1], "4g": l150[1:5], "16g": l150[:16], "4g_l250": l250[:4],
             "novar": no_variants(synth.make_groups(23, 3, n_reads=60, n_haps=3, hap_len=700))}
    i0, u0, r0 = gpu.graph_counters()
    calls = 0
    for name, groups in cases.items():
        batch = abi.Batch(groups)
        want, _ = O.oracle_genotype(batch, gpu.params, n_threads=8)
        for packed in (None, abi.PackedBatch(groups, gpu.lib)):
            ref, got, _ = run_both(gpu, batch, packed)
            calls += 1
            same_results(batch, ref, got)
            errs = compare_results(batch, want, got)
            assert not errs, f"{name} packed={packed is not None}\n" + "\n".join(errs[:20])
    # batches without pairs: no groups at all, and a group without reads (plain and packed)
    g0 = [abi.Group(haps=[b"ACGTACGTACGGTTACA" * 4], reads=[], quals=[], names=[], variants=[])]
    for groups in ([], g0):
        batch = abi.Batch(groups)
        for packed in (None, abi.PackedBatch(groups, gpu.lib)):
            ref, got, st = run_both(gpu, batch, packed)
            calls += 1
            assert st.n_pairs == 0
            assert np.array_equal(ref.grp_mid_occ[:batch.n_groups], got.grp_mid_occ[:batch.n_groups])
    i1, u1, r1 = gpu.graph_counters()
    assert r1 - r0 == calls and (i1 - i0) + (u1 - u0) == calls
    # at most one instantiation per topology: plain / packed x (150 bases, 250 bases, no variants), and four without pairs
    assert i1 - i0 <= 10


@pytest.mark.gpu
def test_one_executable_per_topology():
    """shapes A and B differ in topology (read length selects the chain workspace); A, B, A, B instantiates two
    executables and updates them, and a batch of another size with A's topology updates A's"""
    from lancet2_b200.realign import GpuRealigner
    a = abi.Batch(synth.make_region_groups(31, ref_len=6_000)[:1])
    b = abi.Batch(synth.make_region_groups(32, ref_len=6_000, read_len=250)[:1])
    a4 = abi.Batch(synth.make_region_groups(33, ref_len=20_000)[:4])
    g = GpuRealigner(0)
    try:
        assert g.graph_counters() == (0, 0, 0)
        g.set_graph_mode(True)
        first = {}
        for name, batch in (("a", a), ("b", b), ("a", a), ("b", b)):
            res, _ = g.genotype_batch(batch)
            if name in first:
                same_results(batch, first[name], res)
            else:
                first[name] = res
        assert g.graph_counters() == (2, 2, 4)
        res, _ = g.genotype_batch(a4)
        assert g.graph_counters() == (2, 3, 5)
        want, _ = O.oracle_genotype(a4, g.params, n_threads=8)
        assert not compare_results(a4, want, res)
    finally:
        g.close()


@pytest.mark.gpu
def test_overflow_pass_in_graph_mode():
    """reads inside a tandem repeat with a large fixed mid_occ take the host-driven overflow pass after the graph"""
    from lancet2_b200.realign import GpuRealigner
    from test_gpu_packed import homopolymer_group
    prm = O.default_params()
    prm.mid_occ = 100000
    rng = np.random.default_rng(404)
    groups = [homopolymer_group(rng, 300, 6), synth.make_group(rng, n_reads=40, n_haps=3, hap_len=500)]
    batch = abi.Batch(groups)
    want, wst = O.oracle_genotype(batch, prm, n_threads=8)
    g = GpuRealigner(0, params=prm)
    try:
        g.set_graph_mode(True)
        for packed in (None, abi.PackedBatch(groups, g.lib)):
            got, st = g.genotype_packed(packed, batch) if packed is not None else g.genotype_batch(batch)
            errs = compare_results(batch, want, got)
            assert not errs, "\n".join(errs[:20])
            assert st.reserved > 0  # pairs that went through the overflow pass
            assert (st.n_anchors, st.chain_evals, st.n_aligned) == (wst.n_anchors, wst.chain_evals, wst.n_aligned)
        assert g.graph_counters()[2] == 2
    finally:
        g.close()


@pytest.mark.gpu
def test_group_status_in_graph_mode():
    """a pair beyond 65,535 anchors fails its own group with the same codes as in stream mode"""
    from lancet2_b200.realign import GpuRealigner, LgrError
    from test_gpu_packed import homopolymer_group
    prm = O.default_params()
    prm.mid_occ = 1000000
    rng = np.random.default_rng(11)
    bad = homopolymer_group(rng, 1200, 2, read_len=1000, flank=200)
    bad = abi.Group(haps=bad.haps, reads=[bad.haps[0][195:1195]], quals=[bytes([30] * 1000)], names=["bad"], variants=bad.variants)
    ok1 = synth.make_group(rng, n_reads=50, n_haps=3, hap_len=600)
    ok2 = synth.make_group(rng, n_reads=30, n_haps=2, hap_len=400)
    batch = abi.Batch([ok1, bad, ok2])
    g = GpuRealigner(0, params=prm)
    try:
        ref, _ = g.genotype_batch(batch, group_status=True)
        g.set_graph_mode(True)
        with pytest.raises(LgrError) as ei:
            g.genotype_batch(batch)
        assert ei.value.code == abi.LGR_E_LIMIT
        res, _ = g.genotype_batch(batch, group_status=True)
        assert res.rc == ref.rc == abi.LGR_E_PARTIAL
        assert res.grp_status[:3].tolist() == ref.grp_status[:3].tolist() == [0, abi.LGR_E_LIMIT, 0]
        assert res.assign[:batch.n_assign].tobytes() == ref.assign[:batch.n_assign].tobytes()
        # the context keeps working after the failed call
        good = abi.Batch([ok1, ok2])
        want, _ = O.oracle_genotype(good, prm, n_threads=8)
        assert not compare_results(good, want, g.genotype_batch(good)[0])
    finally:
        g.close()


@pytest.mark.gpu
def test_switching_modes_and_stage_times(gpu):
    """off / on / off / on on one context gives the same results; lgr_run_resident follows the mode; the stage times
    come from event-record nodes of the graph"""
    groups = synth.make_region_groups(41, ref_len=12_000)[:6]
    batch = abi.Batch(groups)
    ref, _ = gpu.genotype_batch(batch)
    for on in (True, False, True, False):
        gpu.set_graph_mode(on)
        res, st = gpu.genotype_batch(batch)
        same_results(batch, ref, res)
        if on:
            stages = (st.ms_k_index, st.ms_k_sketch, st.ms_k_map, st.ms_k_ext, st.ms_k_assign)
            assert st.ms_kernels > 0 and all(t > 0 for t in stages), (st.ms_kernels, stages)
            assert sum(stages) <= st.ms_kernels * 1.001 + 1e-3
    gpu.upload(batch)
    gpu.set_graph_mode(True)
    try:
        r0 = gpu.graph_counters()[2]
        st = gpu.run_resident()
        st = gpu.run_resident()
        assert gpu.graph_counters()[2] == r0 + 2 and st.ms_kernels > 0
        same_results(batch, ref, gpu.download(batch))
    finally:
        gpu.set_graph_mode(False)


@pytest.mark.gpu
def test_adapter_direct_graph_equals_stream_mode():
    """Genotype() from 8 threads, all on direct contexts, with GenotypeBatcher::Options::direct_graph off and on:
    the same evidence, and every call of the graph run launched a graph"""
    lib = _lib()
    lib.lgr_adapter_direct_graph_run.argtypes = [C.c_int, C.POINTER(abi.LgrBatchIn), C.c_char_p, C.c_char_p] + \
        [C.c_void_p] * 6 + [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p, C.c_longlong]
    lib.lgr_adapter_direct_graph_run.restype = C.c_int
    groups = synth.make_region_groups(51, ref_len=60_000)[:16] + synth.make_groups(52, 4, n_reads=96, n_haps=4, hap_len=800, read_len=250)
    batch = abi.Batch(groups)
    names = [nm for g in groups for nm in g.names]
    hs = np.asarray([abi.x31_hash(nm) for nm in names], dtype=np.uint64)
    cols = (np.asarray([0 if nm.startswith("n") else 1 for nm in names], dtype=np.int32), (10_000 + hs % 10_000).astype(np.int64),
            ((hs // 7 % 1000).astype(np.int64) - 500), ((hs // 3 % 2) * 0x10 + (hs // 5 % 2) * 0x2).astype(np.uint16),
            (hs // 11 % 61).astype(np.uint8), (hs // 13 % 2).astype(np.uint8))
    blob = b"\0".join(x.encode() for x in names) + b"\0"
    bi = batch.c_struct()
    rounds = 2
    dumps = []
    for graph in (0, 1):
        counters = np.zeros(22, dtype=np.uint64)
        buf = C.create_string_buffer(64 << 20)
        n = lib.lgr_adapter_direct_graph_run(0, C.byref(bi), blob, b"normal\0tumor\0", *[c.ctypes.data for c in cols], 8, rounds,
                                             graph, counters.ctypes.data, buf, len(buf))
        assert n > 0, buf.value.decode()
        assert int(counters[1]) == rounds * len(groups)
        assert int(counters[21]) == (rounds * len(groups) if graph else 0)
        dumps.append(buf.value)
    assert dumps[0] == dumps[1]
