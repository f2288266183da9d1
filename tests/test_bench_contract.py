"""The driver depends on bench.py's one-line JSON contract.  The reference arm (--impl reference) needs no GPU, so its
line is checked here on the CPU; the GPU arm's line is checked in test_bench_contract_gpu (marker gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import rvtest as T

BENCH = os.path.join(T.ROOT, "bench.py")
COMMON = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
          "dtype", "data", "config", "e2e"}


def _one_line(args, timeout):
    r = subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _one_line(["--impl", "reference", "--steps", "1", "--warmup", "0"], 600)
    assert COMMON <= set(d) and d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["value"] > 10 and "workload" in d["config"] and d["vs_baseline"] is None and d["dtype"] == "f64"


def _dumped(path):
    return {n: np.load(os.path.join(str(path), n + ".npy")) for n in ("logp", "status")}


def test_reference_arm_dumps_its_last_step(tmp_path):
    """--dump-outputs: logp / status of the LAST timed step as float64, identical from run to run with the same arguments."""
    runs = []
    for k in range(2):
        _one_line(["--impl", "reference", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path / str(k))], 600)
        runs.append(_dumped(tmp_path / str(k)))
    assert sorted(os.listdir(str(tmp_path / "0"))) == ["logp.npy", "status.npy"]
    a, b = runs
    assert a["logp"].dtype == np.float64 and a["status"].dtype == np.float64 and a["logp"].shape == a["status"].shape == (4096,)
    assert np.array_equal(a["status"], b["status"]) and np.array_equal(a["logp"], b["logp"])
    # the checker build of the oracle on the walkers of step 1 (the last of two)
    lo, so, _ = T.orc_logp_batch(np.zeros((2, 7)), T.FP10, T.FE10, 2.0, T.load_vels("HD155358.vels"), bench.walker_ball(4096, 1235))
    ok = so == 0
    assert np.array_equal(a["status"], so) and ok.mean() > 0.9 and np.abs(a["logp"][ok] - lo[ok]).max() < 1e-6


def test_dump_outputs_samples_a_large_batch(tmp_path):
    n = bench.DUMP_SAMPLE + 12345
    logp, status = -np.arange(n, dtype=np.float64), (np.arange(n) % 3).astype(np.int32)
    for k in range(2):
        bench.dump_outputs(str(tmp_path / str(k)), logp, status)
    files = sorted(os.listdir(str(tmp_path / "0")))
    assert files == ["logp.npy", "status.npy", "walker_index.npy"]
    assert sum(os.path.getsize(str(tmp_path / "0" / f)) for f in files) <= 64 << 20
    idx = np.load(str(tmp_path / "0" / "walker_index.npy"))
    assert np.array_equal(idx, np.load(str(tmp_path / "1" / "walker_index.npy")))        # a fixed sample
    idx = idx.astype(np.int64)
    assert len(idx) == bench.DUMP_SAMPLE and (np.diff(idx) > 0).all() and idx[-1] < n
    d = _dumped(tmp_path / "0")
    assert np.array_equal(d["logp"], logp[idx]) and np.array_equal(d["status"], status[idx])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, BENCH, "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def _check_gpu_dump(path, W, seed, ok_fraction):
    """The dumped last step against the checker oracle on its first 256 walkers (bench.py seeds step s with 1000 + s)."""
    d = _dumped(path)
    assert d["logp"].dtype == np.float64 and d["status"].dtype == np.float64 and d["logp"].shape == d["status"].shape == (W,)
    ok = d["status"] == 0
    assert ok.mean() == ok_fraction and np.isneginf(d["logp"][~ok]).all()
    lo, so, _ = T.orc_logp_batch(np.zeros((2, 7)), T.FP10, T.FE10, 2.0, T.load_vels("HD155358.vels"),
                                 bench.walker_ball(W, seed)[:256])
    okm = so == 0
    assert np.array_equal(d["status"][:256], so) and np.abs(d["logp"][:256][okm] - lo[okm]).max() < 1e-6


@pytest.mark.gpu
def test_gpu_arm_one_step_without_warmup(tmp_path):
    """--steps sets the number of timed steps, down to one step without warm-up (the CPU baseline still has its inputs)."""
    d = _one_line(["--steps", "1", "--warmup", "0", "--walkers", "4096", "--cpu-sample", "64", "--no-ess", "--no-var",
                   "--dump-outputs", str(tmp_path)], 600)
    assert d["steps"] == 1 and d["warmup"] == 0 and d["gpu_launches"] == 5 and d["cpu_baseline"]["parity_status_equal"]
    _check_gpu_dump(tmp_path, 4096, 1000, d["config"]["ok_fraction"])


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    d = _one_line(["--steps", "3", "--warmup", "3", "--walkers", "8192", "--cpu-sample", "256", "--ess-rows", "60",
                   "--ess-budget", "4,3,4", "--dump-outputs", str(tmp_path)], 900)
    _check_gpu_dump(tmp_path, 8192, 1005, d["config"]["ok_fraction"])
    assert COMMON <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] == 3 and d["scaling"] == "weak" and d["dtype"] == "f64"
    assert d["gpu_launches"] == 15 and d["value"] > 1e5          # 3 steps x (3 item-order kernels + likelihood + finalize)
    assert d["e2e"]["h2d_bytes_per_step"] == 8192 * 80 and d["e2e"]["d2h_bytes_per_step"] == 8192 * 12 and d["e2e"]["value"] > 1e5
    rf = d["roofline"]
    assert rf["bound"] == "fp64_fma_pipe" and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-12 and rf["unit"] == "TFLOP/s"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["parity_status_equal"] and cb["parity_max_abs_logp_diff"] < 1e-6
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    # side blocks: ESS/s of the three samplers from the equilibrated ensemble, the variational kernel, profile-sourced figures
    for k in ("stretch", "mh", "smala"):
        assert d["ess"][k]["ess_per_s"] > 0 and d["ess"][k]["recorded_rows"] >= 50 and 0.05 < d["ess"][k]["accept_rate"] < 0.95
    assert d["var"]["value"] > 1e3 and 0 < d["var"]["roofline"]["frac"] < 1.2
    assert rf["from_profile"]["file"] == "profiles/roofline_inputs.json" and "source" in rf["from_profile"]["loglik_kernel"]
