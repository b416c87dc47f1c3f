"""bench.py's host-side arithmetic (no GPU): SURVEY.md 8(d)'s algorithmic bytes and the profiler-derived block that
the bench line quotes from profiles/*_metrics.json instead of typed-in constants."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _words_from_halves(h):
    return h[:, 0].astype(np.uint64) | (h[:, 1].astype(np.uint64) << np.uint64(32))


def test_algorithmic_bytes_formulas():
    W, A, Q, n = 781, 456, 4, 1 << 19
    ntt, merkle = bench.algorithmic_bytes(W, A, Q, n, 1, 4)
    assert ntt == 8 * W * n * 4 + 8 * A * n * 4 + 8 * Q * n * 3
    assert merkle == sum(8 * c * n * 2 + 32 * (2 * n * 2 - 16) for c in (W, A, Q))
    # the dominant launch group of the bench line: trace tree of a config-2 proof
    assert 8 * W * (2 * n) + 32 * (2 * 2 * n - 16) == 6618611200
    assert bench.rows_for(1024) == 1 << 19 and bench.rows_for(1) == 1 << 16 and bench.rows_for(8192) == 1 << 22


def test_profile_metrics_are_read_from_the_committed_capture():
    m = bench.profile_metrics()
    assert m is not None and m["_file"].startswith("profiles/") and m.get("commit") and m.get("date")
    with open(os.path.join(ROOT, "profiles", "current_metrics.json")) as f:
        assert json.load(f)["file"] == os.path.basename(m["_file"])
    p = bench.leaf_hash_profile(m, 98 * (1 << 20))
    assert p is not None and "leaf_hash" in p["source"]
    # DRAM traffic of the captured launch is within 2 % of the algorithmic bytes (no re-reads), and the instruction
    # count per permutation is what DESIGN.md 4.1 quotes
    assert abs(p["dram_bytes_per_launch"] / 6618611200 - 1) < 0.02
    assert 15e3 < p["thread_instructions_per_permutation"] < 30e3
    assert 0 < p["issue_active"] <= 1 and 0 < p["alu_pipe_busy"] <= 1


def test_workload_config_names_the_baseline_workload():
    class A:
        instances, gpus = 1024, 1
    c = bench.workload_config(A)
    assert c["trace_rows"] == 1 << 19 and c["trace_columns"] == 781 and "1024 scalar-muls" in c["workload"]
    assert "model" not in c


def test_dumped_words_are_exact_and_the_dump_is_bounded(tmp_path, monkeypatch):
    w = np.array([0, 1, 0xFFFFFFFF, 1 << 32, 0xFFFFFFFF00000000, 0xFFFFFFFFFFFFFFFF], dtype=np.uint64)
    h = bench.u64_as_f64_halves(w)
    assert h.dtype == np.float64 and h.shape == (6, 2) and (_words_from_halves(h) == w).all()
    bench.dump_outputs(str(tmp_path / "d"), {"proof_words": h})
    assert (np.load(tmp_path / "d" / "proof_words.npy") == h).all()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", h.nbytes - 1)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "e"), {"proof_words": h})
    assert not (tmp_path / "e").exists()


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_proof(gpu_ctx, tmp_path):
    """bench.py --dump-outputs writes what its last timed step returned: step i proves batch i % 3 (seed
    config_seed(2) + b on rank 0), so with --steps 2 that is batch 1, whose pb254_prove proof and native results
    the dumped arrays must equal exactly."""
    from plonky2_bn254_b200 import inputs as I
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--instances", "3", "--no-cpu-baseline", "--no-other-configs", "--no-pipelined",
                        "--dump-outputs", str(out)], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    inp, ts = I.make_inputs(I.KIND_G1, 3, I.config_seed(2) + 1)
    pf = gpu_ctx.prove(I.KIND_G1, inp, ts)
    words = _words_from_halves(np.load(out / "proof_words.npy"))
    assert words.size == pf.words().size and (words == pf.words()).all()
    assert (np.load(out / "results.npy") == pf.results().reshape(3, -1)).all()
