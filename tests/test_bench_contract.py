"""bench.py prints ONE JSON line with the keys the driver reads (task contract): the reference arm on the CPU here, the
B200 arm on a GPU box with a small shard."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def run_bench(*args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=timeout, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_prints_the_contract_line():
    lines = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-rows", "20000")
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert BASE_KEYS <= set(j) and j["impl"] == "reference" and j["unit"] == "examples/s" and j["higher_is_better"] is True
    assert j["value"] > 0 and j["gpu_launches"] == 0 and "workload" in j["config"]
    cb = j["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] == "port" and cb["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "examples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    assert run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0", "--cpu-rows", "20000",
                     env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_reference_arm_uses_every_host_thread_under_torchrun():
    """torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm must still use the host's cores (VERDICT r1)."""
    lines = run_bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", "--cpu-rows", "20000",
                      env={"RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0", "OMP_NUM_THREADS": "1"})
    assert len(lines) == 1
    cb = json.loads(lines[0])["cpu_baseline"]
    n = len(os.sched_getaffinity(0))
    assert cb["host_threads"] == n and cb["cores"] in (n, max(1, n // 2), max(1, n // 4)) and len(cb["runs_seconds"]) == 3


def load_dump(out_dir):
    import numpy as np
    return {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in ("weights", "loss_history")}


def test_reference_arm_dumps_the_outputs_of_every_step(tmp_path):
    """--steps sets the number of timed iterations; --dump-outputs writes what the timed run returned, the same on every run."""
    for k in ("a", "b"):
        lines = run_bench("--impl", "reference", "--steps", "6", "--warmup", "0", "--cpu-rows", "20000", "--dim", "64",
                          "--dump-outputs", str(tmp_path / k))
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 6
    a, b = load_dump(tmp_path / "a"), load_dump(tmp_path / "b")
    assert a["weights"].shape == (64,) and a["loss_history"].shape == (6,)
    for n in a:
        assert a[n].dtype == b[n].dtype == "float64" and (a[n] == b[n]).all()


@pytest.mark.gpu
def test_b200_arm_prints_the_contract_line(tmp_path):
    lines = run_bench("--rows", "400000", "--steps", "4", "--warmup", "3", "--cpu-rows", "20000",
                      "--dump-outputs", str(tmp_path))
    assert len(lines) == 1
    j = json.loads(lines[0])
    out = load_dump(tmp_path)
    assert out["weights"].shape == (1024,) and out["weights"].dtype == "float64" and out["loss_history"].shape == (4,)
    assert out["loss_history"][-1] == j["final_loss"]
    assert BASE_KEYS | {"roofline", "clocks"} <= set(j) and "impl" not in j
    assert j["n_gpus"] == 1 and j["steps"] == 4 and j["warmup"] == 3 and j["dtype"] == "f64" and j["data"] == "synthetic"
    assert j["scaling"] in ("strong", "weak") and j["vs_baseline"] is None and j["value"] > 0 and j["gpu_launches"] > 0
    r = j["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm" and r["unit"] == "GB/s"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert {"value", "unit", "cores", "kind", "sample"} <= set(j["cpu_baseline"])
    e = j["e2e"]
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(e)
    assert e["h2d_bytes_per_step"] >= 400000 * 1024 * 4 / 4 and e["d2h_bytes_per_step"] > 0 and 0 < e["value"] < j["value"]
    # the accounting of pass fusion is explicit
    assert j["sweeps"] >= j["passes"] - j["fused_passes"] and j["fused_passes"] == 3
    assert j["unfused"]["loss_history_bit_identical_to_fused"] is True and j["unfused"]["sweeps"] == j["passes"]
    assert j["memoized"]["weights_and_history_bit_identical_to_default"] is True and j["memoized"]["sweeps"] < j["sweeps"]
    assert j["clocks"] is None or {"sm_mhz", "sm_max_mhz", "reasons"} <= set(j["clocks"])
    # the full-workload comparison with the oracle rides in the line itself (north_star: weights within 1e-5)
    p = j["parity"]
    assert p["rows"] == 400000 and p["iters"] == 10 and p["pass"] is True and p["shards_equal_cpu_twin"] is True
    assert p["w_rel_err"] <= 1e-9 and p["max_loss_rel_err"] <= 1e-11 and p["passes_equal"] and p["history_len_equal"]
    assert j["roofline"]["kernel"].startswith("k1_ring_kernel<float")
