"""bench.py contract checks that need no GPU: the reference arm (CPU restatement on the host cores) prints one JSON
line with the keys its readers expect, the declared work counts are consistent, and --dump-outputs splits a chunk into
its vectors and writes them exactly, or as a fixed sample within its size limit."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from oracle.params import Phase1Params

import bench


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--curve", "bls12_377",
                          "--chunk-log", "9"], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["value"] > 0 and line["vs_baseline"] is None
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0


def test_declared_work_counts():
    # the kernels do fewer field multiplications than the reference's double-and-add: b*D + (b/2)*11 (SURVEY.md §8d)
    ref = {"bls12_377": 253 * 7 + 126.5 * 11, "bw6_761": 377 * 7 + 188.5 * 11, "mnt4_753": 753 * 10 + 376.5 * 11}
    for curve, ref_fm in ref.items():
        ours = bench.declared_fq_muls_per_point(curve, 0)
        assert 0.4 * ref_fm < ours < ref_fm
    assert bench.macs_per_fq_mul(12) == 300 and bench.macs_per_fq_mul(24) == 1176 and bench.macs_per_fq_mul(8) == 136


@pytest.mark.parametrize("compressed", [True, False])
@pytest.mark.parametrize("k", [1, 3])
def test_accumulator_vectors_follow_the_chunk_layout(k, compressed):
    o = Phase1Params.new_chunk("mnt6_753", k, 4, 3, 4)          # chunk 3 is a G1-only tail
    (g1c, g2c), (g1u, g2u) = o.sizes(True), o.sizes(False)
    es = {"g1_c": g1c, "g2_c": g2c, "g1_u": g1u, "g2_u": g2u}
    offs = o.offsets(compressed)
    buf = (np.arange(offs[-1]) % 251).astype(np.uint8)
    vecs = bench.accumulator_vectors(buf, {"g1_count": o.g1_count, "other_count": o.other_count}, es, compressed)
    assert [n for n, _ in vecs] == list(bench.VECTOR_NAMES)
    for i, (_, v) in enumerate(vecs):
        assert v.tobytes() == buf[offs[i]:offs[i + 1]].tobytes()
        assert v.shape[1] == es[("g1" if bench.VECTOR_GROUPS[i] == 0 else "g2") + ("_c" if compressed else "_u")]


def test_dump_outputs_exact_then_sampled_within_budget(tmp_path, monkeypatch):
    rnd = np.random.default_rng(1)
    arrays = [("a", rnd.integers(0, 256, (1000, 48), dtype=np.uint8)), ("b", rnd.integers(0, 256, (1, 96), dtype=np.uint8))]
    bench.dump_outputs(str(tmp_path / "whole"), arrays)
    assert sorted(os.listdir(tmp_path / "whole")) == ["a.npy", "b.npy"]
    for name, a in arrays:
        got = np.load(tmp_path / "whole" / (name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, a)
    monkeypatch.setattr(bench, "DUMP_BUDGET", 100_000)
    for run in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / run), arrays)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= 100_000
        for name, a in arrays:
            rows = np.load(tmp_path / run / (name + "_rows.npy"))
            assert rows.dtype == np.float64 and 1 <= len(rows) < 1000 and np.all(np.diff(rows) > 0)
            assert np.array_equal(np.load(tmp_path / run / (name + ".npy")), a[rows.astype(np.int64)])
    for f in os.listdir(tmp_path / "s1"):
        assert np.array_equal(np.load(tmp_path / "s1" / f), np.load(tmp_path / "s2" / f))
