"""CPU: bench.py's reference arm (the oracle port of the reference's CPU path) prints one JSON line with the
contract's keys; the CUDA arm cannot run without a GPU and must say so loudly."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    sys.path.insert(0, ROOT)
    import bench
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-fit", "3,4,5"], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "proofs/s" and line["value"] > 0
    # one worker per USABLE core (affinity mask / cgroup quota), not per os.cpu_count(); the value is an extrapolation
    # through the fitted cost model and says so
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] == bench.usable_cores()
    assert line["extrapolated"] is True and line["cpu_baseline"]["usable_cores"] == bench.usable_cores()
    fit = line["cpu_baseline"]["fit"]
    assert fit["a_s_per_gate"] >= 0 and fit["b_s_per_gate_log_gate"] >= 0 and fit["extrapolated_s_per_proof"] > 0
    assert set(line["cpu_baseline"]["seconds_per_proof_per_worker"]) == {"3", "4", "5"}
    one = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--cpu-fit", "3,4,5", "--cpu-procs", "1"], capture_output=True, text=True,
                         timeout=300, cwd=ROOT)
    single = json.loads(one.stdout.strip().splitlines()[-1])
    assert single["cpu_baseline"]["cores"] == 1 and 0 < single["value"] <= line["value"] * 1.5
    assert bench.fit_cost([(8, 8.0), (16, 16.0), (32, 32.0)])[0] == __import__("pytest").approx(1.0, rel=1e-6)
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["vs_baseline"] is None
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=60, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_holds_the_proof_words_exactly(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    import numpy as np
    raw = bytes.fromhex(json.load(open(os.path.join(ROOT, "tests", "golden", "proof_2p20.json")))["proof_hex"])
    other = bytes(reversed(raw))
    bench.dump_outputs(str(tmp_path / "out"), [raw, other])
    got = np.load(tmp_path / "out" / "proof.npy")
    assert got.dtype == np.float64 and got.shape == (2, 24, 8)
    for lane, proof in enumerate((raw, other)):
        words = [sum(int(got[lane, k, i]) << (32 * i) for i in range(8)) for k in range(24)]
        assert words == [int.from_bytes(proof[i:i + 32], "big") for i in range(0, 768, 32)]


def test_cuda_arm_refuses_without_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0  # no CPU fallback: the product arm must fail, not silently measure something else
