"""bench.py --dump-outputs: what the last timed step computed, as float .npy files, so that two builds (or the GPU path and
the CPU oracle) can be compared output for output on the same seeded workload."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

import bench
from polypolish_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".npy")}


def _bench(out_dir, *extra):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "50kbp_x100", "--dump-outputs", str(out_dir)] + list(extra),
                       cwd=ROOT, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr[-2000:]
    return json.loads([l for l in p.stdout.splitlines() if l.startswith("{")][-1])


def test_dump_outputs_whole_result(tmp_path):
    seqs = [b"ACGT", b"", b"GGA"]
    names = bench.dump_outputs(tmp_path, seqs, [1, 0, 2], [0, 4, 0], [10.5, 0.0, 7.25], 9)
    got = _load(tmp_path)
    assert sorted(got) == names == ["changed", "contig_offsets", "n_aln_used", "polished_bases", "total_depth", "zero_depth"]
    assert got["polished_bases"].dtype == np.float32 and bytes(got["polished_bases"].astype(np.uint8)) == b"ACGTGGA"
    assert all(a.dtype == np.float64 for k, a in got.items() if k != "polished_bases")
    assert got["contig_offsets"].tolist() == [0, 4, 4, 7]
    assert got["changed"].tolist() == [1, 0, 2] and got["zero_depth"].tolist() == [0, 4, 0]
    assert got["total_depth"].tolist() == [10.5, 0.0, 7.25] and got["n_aln_used"].tolist() == [9]


def test_dump_outputs_samples_a_large_result_at_fixed_positions(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_FULL_BASES", 1000)
    monkeypatch.setattr(bench, "DUMP_SAMPLE_BASES", 100)
    rng = np.random.default_rng(5)
    seqs = [bytes(rng.choice(list(b"ACGT"), n).astype(np.uint8)) for n in (700, 900)]
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(a, seqs, [0, 0], [0, 0], [1.0, 2.0], 3)
    bench.dump_outputs(b, seqs, [0, 0], [0, 0], [1.0, 2.0], 3)
    ga, gb = _load(a), _load(b)
    idx = ga["polished_bases_index"].astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and idx[-1] < 1600
    assert bytes(ga["polished_bases"].astype(np.uint8)) == bytes(np.frombuffer(b"".join(seqs), np.uint8)[idx])
    assert all(np.array_equal(ga[k], gb[k]) for k in ga)


def test_dump_outputs_stays_under_its_limit():
    """The largest dump either way (whole bases or a sample with its positions), with room for 10^5 contigs' statistics."""
    per_contig = 100_000 * 4 * 8
    assert 4 * bench.DUMP_FULL_BASES + per_contig <= bench.DUMP_MAX_BYTES
    assert 12 * bench.DUMP_SAMPLE_BASES + per_contig <= bench.DUMP_MAX_BYTES


def test_fasta_sequences_of_the_oracle(oracle):
    with tempfile.TemporaryDirectory() as d:
        syn = api.Synth(seed=3, n_contigs=3, contig_len=20_000, depth=30)
        fa, sams = syn.write(d)
        r = oracle.polish(fa, sams)
    seqs = bench.fasta_sequences(r["fasta"])
    assert [len(s) for s in seqs] == r["new_length"]
    assert sum(r["changed"]) > 0


def test_bench_reference_dump(tmp_path):
    """--impl reference dumps the oracle's result for the same seeded workload; two runs write the same arrays."""
    runs = []
    for name in ("a", "b"):
        line = _bench(tmp_path / name, "--impl", "reference", "--steps", "2", "--warmup", "0")
        assert line["steps"] == 2 and line["config"]["same_config"]
        runs.append(_load(tmp_path / name))
    assert "polished_bases_index" not in runs[0] and len(runs[0]["polished_bases"]) == runs[0]["contig_offsets"][-1]
    assert sorted(runs[0]) == sorted(runs[1]) and all(np.array_equal(runs[0][k], runs[1][k]) for k in runs[0])


@pytest.mark.gpu
def test_bench_dump_matches_the_oracle(tmp_path):
    """The kernel path's last timed step, as bench.py writes it, against the oracle's result on the same workload."""
    line = _bench(tmp_path / "gpu", "--steps", "3", "--warmup", "3", "--no-t3", "--no-cpu-baseline")
    assert line["steps"] == 3
    _bench(tmp_path / "ref", "--impl", "reference", "--steps", "1", "--warmup", "0")
    gpu, ref = _load(tmp_path / "gpu"), _load(tmp_path / "ref")
    assert sorted(gpu) == sorted(ref)
    for k in ("polished_bases", "contig_offsets", "changed", "zero_depth", "n_aln_used"):
        assert np.array_equal(gpu[k], ref[k]), k
    assert ref["changed"].sum() > 0
    # per-position depths are the reference's exactly; their per-contig sum is accumulated in parallel on the device
    np.testing.assert_allclose(gpu["total_depth"], ref["total_depth"], rtol=1e-12)
