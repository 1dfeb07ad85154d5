"""The committed bench lines (profiles/r0*_bench_n*.json, written by bench.py on a B200) carry every key
the measurement contract names; bench.py's CLI parses the driver's flags and --dump-outputs writes the
last step's arrays.  No GPU needed except for the test marked gpu."""
import json
import os
import subprocess
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _line(name):
    with open(os.path.join(ROOT, "profiles", name)) as f:
        return json.load(f)


def test_bench_line_has_the_contract_keys():
    d = _line("r01_bench_n1.json")
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks",
              "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["higher_is_better"] is True
    assert "workload" in d["config"] and "model" not in d["config"]
    r = d["roofline"]
    for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r, k
    assert r["bound"] in ("hbm", "tensor") and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert 0.5 < r["traffic"] / r["algorithmic_bytes_per_launch"] < 1.5      # no wasted re-reads
    s = r["second_kernel"]
    assert s["bound"] == "tensor" and 0 < s["frac"] < 1
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}


def test_eight_gpu_line_is_the_whole_job_aggregate():
    d1, d8 = _line("r01_bench_n1.json"), _line("r01_bench_n8.json")
    assert d8["n_gpus"] == 8 and d8["metric"] == d1["metric"] and d8["unit"] == d1["unit"]
    assert d8["config"]["population"] == 8 * d1["config"]["population"]
    assert 6.0 < d8["value"] / d1["value"] < 8.5
    assert "cpu_baseline" not in d8                     # rank 0 at N=1 only


def test_bench_cli_accepts_the_driver_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--help"], capture_output=True, text=True)
    assert out.returncode == 0
    for flag in ("--gpus", "--steps", "--warmup", "--impl", "--dump-outputs"):
        assert flag in out.stdout


def test_dump_outputs_writes_the_last_steps_arrays(tmp_path):
    import numpy as np
    import torch

    import bench
    from coevonet_b200 import layout
    pitch = {r: layout.fc_pitch(layout.OBS_DIM[r]) for r in bench.ROLES}
    eng = types.SimpleNamespace(
        last_eval=lambda: (1.5, -2.0, 0.25),
        rewards={r: torch.arange(4, dtype=torch.float64) for r in bench.ROLES},
        fitness={r: torch.arange(8, dtype=torch.float64) for r in bench.ROLES},
        theta={r: torch.ones(pitch[r]) for r in bench.ROLES},
        last_delta={r: torch.full((pitch[r],), 0.5) for r in bench.ROLES})
    bench.dump_outputs(eng, str(tmp_path / "out"))
    files = sorted(p.name for p in (tmp_path / "out").iterdir())
    assert files == sorted(["eval_rewards.npy"] + [f"{k}_{r}.npy" for r in bench.ROLES
                                                   for k in ("rewards", "fitness", "theta", "delta")])
    assert np.load(tmp_path / "out" / "eval_rewards.npy").tolist() == [1.5, -2.0, 0.25]
    for r in bench.ROLES:
        theta = np.load(tmp_path / "out" / f"theta_{r}.npy")
        assert theta.dtype == np.float32 and theta.shape == (layout.fc_dim(layout.OBS_DIM[r]),)
        assert np.load(tmp_path / "out" / f"fitness_{r}.npy").dtype == np.float64
    assert sum(p.stat().st_size for p in (tmp_path / "out").iterdir()) < 64 << 20


@pytest.mark.gpu
def test_dump_outputs_of_a_real_engine_are_consistent_and_repeat(tmp_path):
    """bench.dump_outputs on the bench's own engine (small population): the arrays are what the last
    generation produced, and a second run with the same arguments writes the same bits."""
    import numpy as np
    import torch

    import bench
    from coevonet_b200 import engine, layout
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    P = 64

    def run(out):
        torch.manual_seed(0)
        theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in bench.ROLES}
        eng = engine.ESEngine(bench._args_bag(P), torch.device("cuda", 0), theta, comm=engine.Comm())
        eng.step(sync=False)
        before = {r: eng.theta[r].cpu().numpy() for r in bench.ROLES}
        eng.step(sync=False)
        eng.check_status()
        bench.dump_outputs(eng, str(out))
        assert np.load(out / "eval_rewards.npy").tolist() == list(eng.last_eval())
        return before

    before = run(tmp_path / "a")
    run(tmp_path / "b")
    for f in sorted((tmp_path / "a").iterdir()):
        assert np.array_equal(np.load(f), np.load(tmp_path / "b" / f.name)), f.name
    for r in bench.ROLES:
        d = layout.fc_dim(layout.OBS_DIM[r])
        load = lambda k: np.load(tmp_path / "a" / f"{k}_{r}.npy")
        rewards, fitness, theta, delta = load("rewards"), load("fitness"), load("theta"), load("delta")
        assert rewards.shape == fitness.shape == (P,) and theta.shape == delta.shape == (d,)
        assert np.array_equal(fitness, rewards.astype(np.float32).astype(np.float64))   # no fitness sharing
        assert np.array_equal(theta, before[r][:d] + delta)                              # theta += delta
        assert np.abs(delta).max() > 0


def test_bench_rejects_a_step_count_below_one():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True)
    assert out.returncode != 0 and "--steps" in out.stderr


def test_round2_line_carries_parity_secondary_and_floors():
    d = _line("r02_bench_n1.json")
    p = d["parity"]
    assert p["members_sampled"] >= 3 * 128 and 0.0 <= p["member_match_frac"] <= 1.0 and p["episode_forks"] >= 0
    fl = d["roofline"]["floors"]
    assert fl["per_launch_hbm_us"] > fl["per_launch_tensor_us"] > 0         # `bound` hbm is the binding floor
    ws = d["roofline"]["whole_step"]
    assert 0.0 < ws["frac_of_hbm_peak"] < 1.0 and "ls_member_tc_kernel" in d["roofline"]["kernel"]
    assert abs(fl["per_rollout_hbm_bytes_streamed"] - 25 * fl["per_rollout_hbm_bytes_if_rows_stayed_on_chip"]) < 1
    assert d["roofline"]["fp32_peak_theoretical_tflops"] >= d["roofline"]["fp32_peak_tflops"] * 0.95
    assert d["e2e"]["steps"] == d["steps"]                                 # e2e over the full --steps, host clock
    s = d["secondary"]
    names = " ".join(k["kernel"] for k in s["kernels"])
    for k in ("K3", "K5", "K6", "K7"):
        assert k in names
    for k in s["kernels"]:
        assert k["us_per_launch"] > 0 and k["rows"] in (1024, 8192)
        if k["bound"] != "alu":
            assert abs(k["frac"] - k["achieved"] / k["peak"]) < 1e-9
    assert s["config3_ga"]["members_per_gpu"] == 8192 and s["config3_ga"]["ms_per_generation"] > 0
    assert [c["frames_per_member"] for c in s["config4_dqn_forward"]] == [1, 4]
    assert s["config5_dqn_es"]["population"] == 4096


def test_round2_multi_gpu_lines_check_the_sharded_run_against_one_gpu():
    d1 = _line("r02_bench_n1.json")
    for n in (2, 8):
        d = _line(f"r02_bench_n{n}.json")
        assert d["n_gpus"] == n and d["sharded_equals_single"] is True
        assert d["sharded_check"]["rewards_bit_identical"] is True
        assert 0.9 * n < d["value"] / d1["value"] < 1.1 * n
        assert d["secondary"]["config3_ga"]["population"] == 8192 * n
