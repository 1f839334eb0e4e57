"""The parts of bench.py's contract that do not need a GPU -- the reference arm prints
exactly one JSON line with the agreed keys (rank 0) or nothing (other ranks), nothing else
reaches stdout, and the helper parsers behave.  On a GPU (-m gpu): what --dump-outputs writes."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_ref(rank):
    env = dict(os.environ, RANK=str(rank), WORLD_SIZE="2", LASER_B200_REF_BUDGET_S="1.5")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                           "--steps", "1", "--warmup", "1"], env=env, capture_output=True, text=True, timeout=600)


def test_reference_arm_rank0_prints_one_json_line():
    out = run_ref(0)
    assert out.returncode == 0, out.stderr
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "TFLOP/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["vs_baseline"] is None


def test_reference_arm_other_ranks_are_silent():
    out = run_ref(1)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_argument_checks():
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=60)
        assert out.returncode == 2 and out.stdout == "", extra


def test_dump_rows_are_a_fixed_sample():
    sys.path.insert(0, ROOT)
    import bench
    rows = bench.dump_rows(8192, 1)
    assert len(rows) == bench.DUMP_ROWS and len(set(rows.tolist())) == bench.DUMP_ROWS and 0 <= rows[0] and rows[-1] < 8192
    assert (rows == bench.dump_rows(8192, 1)).all()
    assert bench.DUMP_ROWS * 8192 * 4 <= 64 << 20


@pytest.mark.gpu
def test_dump_outputs_hold_the_timed_product(tmp_path):
    """--dump-outputs writes the sampled rows of the last timed step's C, and they are the product of the seeded inputs"""
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np
    import oracle as O
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-4000:]
    assert json.loads(out.stdout)["steps"] == 2
    assert os.listdir(tmp_path) == ["C.npy"]
    C = np.load(tmp_path / "C.npy")
    n = bench.MNK
    assert C.dtype == np.float32 and C.shape == (bench.DUMP_ROWS, n)
    pick = np.arange(0, bench.DUMP_ROWS, 255)
    rows = bench.dump_rows(n, 1)[pick]
    A = O.fill_uniform_f32(n * n, 42, -0.1, 0.1).reshape(n, n)
    B = O.fill_uniform_f32(n * n, 43, -0.1, 0.1)
    a = np.ascontiguousarray(A[rows]).reshape(-1)
    want = np.zeros(len(rows) * n, np.float32)
    O.cpu_gemm_strided_f32(len(rows), n, n, 1.0, a, n, 1, B, n, 1, 0.0, want, n, 1)
    assert O.normwise_relative_error(C[pick], want) < 2e-6


def test_clock_sampler_parsing_and_peaks():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.proc = type("P", (), {"terminate": lambda self: None, "wait": lambda self, timeout=None: 0, "kill": lambda self: None})()
    s.lines = ["0, 1965, 1965, 120.5, 0x0, Not Active, Not Active, Not Active, Not Active",
               "0, 1400, 1965, 990.1, 0x4, Not Active, Not Active, Not Active, Active",
               "0, 1380, 1965, 1001.0, 0x4, Not Active, Not Active, Not Active, Active"]
    c = s.stop()
    assert c["sm_max_mhz"] == 1965 and c["reasons"] == ["sw_power_cap"] and 1380 <= c["sm_mhz"] <= 1400
    p = bench.load_peaks()
    assert p["bf16"] > 0 and p["source"] in ("measured", "fallback")
