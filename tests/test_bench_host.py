"""Tests of bench.py: on the CPU its host logic -- workload generation (BASELINE.json configs[1], SURVEY.md
8d "C2"), clock-sample parsing, the reference arm's JSON contract and --dump-outputs on a tiny sample; on the
GPU, --dump-outputs of the engine arm."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_workload_is_deterministic_and_has_the_documented_regime_shares():
    h, z = bench.make_inputs_numpy("hybrid", 400_000)
    h2, z2 = bench.make_inputs_numpy("hybrid", 400_000)
    assert np.array_equal(h, h2) and np.array_equal(z, z2)
    h3, _ = bench.make_inputs_numpy("hybrid", 1000, obs0=400_000)        # another rank's shard: other draws
    assert not np.array_equal(h[:1000], h3)
    assert z.min() >= -5 and z.max() <= 5 and h.min() >= 0.5 and h.max() <= 200
    share = {"sp": np.mean((h > 13) & (h <= 170)), "normal": np.mean(h > 170),
             "alt": np.mean((h > 1) & (h <= 13) & (h != 2)), "devroye": np.mean((h == 1) | (h == 2)),
             "gamma": np.mean(h < 1)}
    # SURVEY.md 8d: 78.6 % / 15 % / 5.8 % / 0.5 % / 0.13 %
    for k, want in (("sp", 0.786), ("normal", 0.15), ("alt", 0.058), ("devroye", 0.005), ("gamma", 0.0013)):
        assert abs(share[k] - want) < 0.1 * want + 0.0006, (k, share[k])
    n, z1 = bench.make_inputs_numpy("pg1", 1000)
    assert n.dtype == np.int32 and np.all(n == 1) and z1.shape == (1000,)


def test_clock_sampler_parsing():
    class Proc:
        def terminate(self):
            pass
    c = bench.ClockSampler.__new__(bench.ClockSampler)
    c.proc = Proc()
    t = time.time()
    ok = ["0", "1965", "1965", "480.1", "0x0", "Not Active", "Not Active", "Not Active", "Not Active"]
    cap = ["0", "1800", "1965", "[N/A]", "0x4", "Not Active", "Not Active", "Not Active", "Active"]
    c.rows = [(t - 5, cap), (t, ok), (t + 0.01, ok), (t + 0.02, cap)]
    out = c.stop(t - 0.5, t + 0.5, t - 10)
    assert out["samples"] == 3 and out["window"] == "timed steps"
    assert out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]
    assert out["power_w_max"] == 480.1
    c.rows = [(t - 5, ok), (t - 4, ok)]                      # nothing inside the timed steps: warm-up window
    out = c.stop(t - 0.5, t + 0.5, t - 10)
    assert out["samples"] == 2 and out["window"].startswith("warm-up")
    c.rows = []
    assert c.stop(t - 0.5, t + 0.5, t - 10)["reasons"] == ["no samples"]


def test_reference_arm_prints_one_json_line_with_the_contract_keys(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1", "--num", "200000", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600)
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout + out.stderr[-500:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pg_draws_per_sec" and d["unit"] == "draws/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": "draws/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["draws_per_gpu_per_step"] == 200000
    # --dump-outputs: the draws of the timed step, as the sampler computed them
    from oracle import loader
    assert os.listdir(tmp_path) == ["omega.npy"]
    x = np.load(tmp_path / "omega.npy")
    h, z = bench.make_inputs_numpy("hybrid", 200000)
    assert x.dtype == np.float64
    assert np.array_equal(x, loader.Oracle(d["cpu_baseline"]["kind"]).rpg_hybrid(h, z, seed=bench.SEED, nthreads=4))


def test_dump_sample_is_fixed_and_spans_the_batch():
    assert bench.dump_index(bench.DUMP_DRAWS) is None
    num = 100_000_000
    idx = bench.dump_index(num)
    k = bench.DUMP_DRAWS
    assert idx.size == k and idx.size * 8 <= 64 << 20
    stratum = np.arange(k, dtype=np.int64)                     # one draw inside each of k equal strata
    assert np.all(stratum * num // k <= idx) and np.all(idx < (stratum + 1) * num // k)
    assert np.array_equal(idx, bench.dump_index(num))
    assert bench.dump_index(num, world=8).size == bench.DUMP_DRAWS // 8


@pytest.mark.gpu
def test_engine_dump_is_the_last_timed_step(engine, tmp_path):
    """bench.py --dump-outputs writes the draws of the last timed step (call id steps - 1), sampled when the
    batch is larger than DUMP_DRAWS."""
    num, steps = bench.DUMP_DRAWS + 1_000_003, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                          "--num", str(num), "--no-extras", "--no-cpu-baseline", "--no-e2e",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout)["steps"] == steps
    h, z = bench.make_inputs_numpy("hybrid", num)
    want = engine.rpg_seeded("hybrid", h, z, seed=bench.SEED, call_id=steps - 1)[bench.dump_index(num)]
    assert np.array_equal(np.load(tmp_path / "omega.npy"), want)


def test_reference_arm_under_torchrun_prints_on_rank_0_only():
    """N > 1: the driver launches both arms under torchrun; rank 0 alone runs the CPU reference and prints,
    the other ranks exit 0 without work."""
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29583",
                          os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1", "--draws", "100000"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-800:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 2 and d["value"] > 0
