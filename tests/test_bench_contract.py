"""bench.py's output contract on the arm that runs without a GPU (--impl reference): exactly one
JSON line on stdout with the keys the driver reads; and the GPU arm must refuse to run without a
device instead of falling back."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "alignments/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_gpu_arm_refuses_without_a_device():
    import torch
    if torch.cuda.is_available():
        return  # on the GPU box the arm runs; the parity suite covers it
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "1"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)
    assert not [l for l in p.stdout.splitlines() if l.strip().startswith("{")]


def test_dump_outputs_are_float64_records_of_the_batch(tmp_path, monkeypatch):
    import bench
    import oracle_lib as O
    from lancet2_b200 import abi, synth
    batch = abi.Batch(synth.make_groups(7, 3, read_len=150, hap_len=600, n_haps=3, n_reads=40))
    res, _ = O.oracle_genotype(batch)
    bench.dump_outputs(str(tmp_path / "all"), res)
    got = {f[:-len(".npy")]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert all(v.dtype == np.float64 for v in got.values())
    assert got["aln_pair"].tolist() == list(range(batch.n_pairs))
    assert got["assign_row"].tolist() == list(range(batch.n_assign))
    for f in ("valid", "score", "rs", "qe", "nm", "n_cigar"):
        assert np.array_equal(got[f"aln_{f}"], res.aln[f][:batch.n_pairs]), f
    for f in ("local_score", "folded_read_pos", "hap_id", "allele", "assigned"):
        assert np.array_equal(got[f"assign_{f}"], res.assign[f][:batch.n_assign]), f
    ops = [op for p in range(batch.n_pairs) for op in res.cigar(p)]
    assert ops and got["cigar_ops"].tolist() == ops and got["aln_n_cigar"].sum() == len(ops)
    # beyond the caps: a fixed seeded sample of rows, the same on every call
    monkeypatch.setattr(bench, "DUMP_PAIRS", batch.n_pairs // 3)
    monkeypatch.setattr(bench, "DUMP_ASSIGN", batch.n_assign // 3)
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), res)
    for f in os.listdir(tmp_path / "s1"):
        assert np.array_equal(np.load(tmp_path / "s1" / f), np.load(tmp_path / "s2" / f)), f
    rows = np.load(tmp_path / "s1" / "aln_pair.npy").astype(np.int64)
    assert len(rows) == batch.n_pairs // 3 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "s1" / "aln_score.npy"), res.aln["score"][rows])
    assert len(np.load(tmp_path / "s1" / "assign_row.npy")) == batch.n_assign // 3
    # a byte limit the whole output does not fit: smaller samples, never more bytes than the limit
    monkeypatch.undo()
    limit = sum(os.path.getsize(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")) // 3
    bench.dump_outputs(str(tmp_path / "small"), res, limit=limit)
    small = {f[:-len(".npy")]: np.load(tmp_path / "small" / f) for f in os.listdir(tmp_path / "small")}
    assert 0 < len(small["aln_pair"]) < batch.n_pairs and 0 < len(small["assign_row"]) < batch.n_assign
    assert sum(v.nbytes for v in small.values()) <= limit
    assert small["aln_n_cigar"].sum() == len(small["cigar_ops"])


@pytest.mark.gpu
def test_gpu_arm_steps_and_dumped_outputs(tmp_path):
    """--steps sets the timed steps of every arm, and --dump-outputs writes what the resident arm's last pass
    computed: the arrays the CPU oracle gives for the same workload, bit for bit"""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "2", "--warmup", "1",
                        "--min-step-ms", "0", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "gpu")],
                       capture_output=True, text=True, timeout=1200)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout)
    assert d["steps"] == 2 and d["config"]["passes_per_step"] == 1
    assert d["config"]["passes_timed"] == 2     # passes the resident arm's timed loop actually ran
    assert d["e2e"]["passes_per_step"] == 1 and d["e2e"]["passes_timed"] == 2
    import bench
    import oracle_lib as O
    from lancet2_b200 import abi
    groups = bench.build_workload("tiny", 42)[0]
    params = abi.LgrParams()
    abi.load_library().lgr_default_params(C.byref(params))
    res, _ = O.oracle_genotype(abi.Batch(groups), params, n_threads=os.cpu_count() or 1)
    bench.dump_outputs(str(tmp_path / "cpu"), res)
    names = sorted(os.listdir(tmp_path / "cpu"))
    assert names == sorted(os.listdir(tmp_path / "gpu"))
    for nm in names:
        want, got = np.load(tmp_path / "cpu" / nm), np.load(tmp_path / "gpu" / nm)
        assert got.dtype == np.float64 and np.array_equal(want, got, equal_nan=True), nm
