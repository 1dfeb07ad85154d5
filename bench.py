#!/usr/bin/env python
"""Bench of the population-evaluation hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this build, N GPUs of one node
    python bench.py --impl reference --steps K --warmup W    # the reference's CPU path (port)

Workload (BASELINE.json configs[1]): Co-ES on simple_adversary_v3, 1024 members
per GPU x 16 env instances x 3 roles, 25-cycle episodes, Philox seed-regenerated
noise.  One "step" = one Co-ES generation of the hot path:
for each role  K5 perturb -> K1 fused rollout -> fitness -> K6 update (+ the
fitness all-gather and delta all-reduce when N > 1), then the 10 evaluation
games.  `value` = world-steps/s over all ranks (1 world step = one physics
step = 3 agent `env.step` calls of the AEC reference); weak scaling (1024
members per GPU).  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

P_PER_GPU = 1024
ENVS = 16
CYCLES = 25
FLOP_PER_WORLD_STEP = 822784          # three MLP forwards, SURVEY.md section 8d
ROLES = ("agent_0", "agent_1", "adversary_0")
METRIC = "mpe_env_steps_per_sec"
UNIT = "world-steps/s"


def _args_bag(P):
    return types.SimpleNamespace(
        algorithm="ES", generations=1, population=P, hof_size=1, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=False,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32",
        save=False, envs_per_member=ENVS, reference_compat=True, init_states="device",
        seed=1870300, plots=False, record_history=False)


def _config(n_gpus):
    return {"workload": "Co-ES simple_adversary_v3 population evaluation (BASELINE configs[1])",
            "population_per_gpu": P_PER_GPU, "population": P_PER_GPU * n_gpus, "envs_per_member": ENVS,
            "roles": 3, "cycles_per_episode": CYCLES,
            "noise": "Philox4x32-10: members materialised from the seed by K5 every generation (never stored "
                     "across generations); the update reads sigma*z back as members - theta (K6, members form)",
            "step": "one generation: 3 x perturb (K5), the three roles' rollouts as ONE lockstep pass "
                    "(cev_mpe_rollout_roles_f32: per role and world step a tensor-core member kernel on a share of the "
                    "SMs beside the tensor-core opponent kernel on the rest, then the environment step), 3 x update "
                    "(K6) + apply, 10 eval games on a high-priority stream; no host round trip inside a generation "
                    "(sigma / reward history / status live on the device)",
            "env_step_definition": "world step (3 agent env.step calls); agent-steps/s = 3 x value",
            "cache": "inputs larger than L2 (3 x 1024 member rows = 1.7 GB per GPU vs 126 MB L2)",
            "parallelism": f"population sharded over {n_gpus} GPU(s)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                power.append(float(r[3]))
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7),
                                  ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def _measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def _k1_traffic():
    """DRAM bytes per K1 launch from the committed ncu capture (profiles/), or null."""
    path = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.isfile(path):
        with open(path) as f:
            return json.load(f)
    return None


# ---------------------------------------------------------------------------
# CPU baseline legs (the oracle as the timed baseline -- never on the product path)
# ---------------------------------------------------------------------------
def _cpu_sample(n_episodes, n_procs):
    import numpy as np
    from oracle import mpe_env, serial_port, weights
    rows = {"agent_0": weights.make_fc_rows(1, 10, 1)[0], "agent_1": weights.make_fc_rows(1, 10, 2)[0],
            "adversary_0": weights.make_fc_rows(1, 8, 3)[0]}
    init = mpe_env.draw_initial_states(n_episodes)
    _, wall = serial_port.timed_sample(rows, init, n_procs)
    return n_episodes * CYCLES / wall, wall


def cpu_baseline_block(budget_s=12.0):
    """Episode-serial port on ONE core (how the reference runs), bounded sample."""
    rate, _ = _cpu_sample(16, 1)                       # calibrate
    n = max(32, min(4096, int(budget_s * rate / CYCLES)))
    value, wall = _cpu_sample(n, 1)
    return {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n} episodes of the same workload (batch-1 torch forward + AEC numpy env, "
                      f"oracle/serial_port.py) in {wall:.1f} s; the reference is single-process"}


def parity_block(dev):
    """Member-level parity of the bench workload against the oracle (the checker, never the thing
    measured): the fraction of sampled config-2 members whose fitness is within 1e-4 relative, and the
    episode fork count.  Runs in the cpu_baseline leg (rank 0, N = 1)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_gpu_parity_r2 import member_match_stats
    st = member_match_stats(n_sample=128, P=P_PER_GPU, E=ENVS)
    st["checked_against"] = "oracle/rollout.py on 3 x 128 full members (16 episodes each) of one generation"
    return st


def run_reference_arm(ns):
    """The reference's CPU implementation of the path (port; /root/reference does not
    travel to the GPU box), all host cores, each step a bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    rate1, _ = _cpu_sample(8, 1)
    per_step = max(cores * 4, min(cores * 64, int(6.0 * rate1 * cores / CYCLES)))
    for _ in range(ns.warmup):
        _cpu_sample(max(cores, per_step // 4), cores)
    t0 = time.perf_counter()
    for _ in range(ns.steps):
        _cpu_sample(per_step, cores)
    wall = time.perf_counter() - t0
    value = ns.steps * per_step * CYCLES / wall
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ns.gpus,
            "steps": ns.steps, "warmup": ns.warmup, "ms_per_step": wall / ns.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": _config(ns.gpus),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{per_step} episodes per step over {cores} processes "
                                       "(oracle/serial_port.py: episode-serial batch-1 port of the reference path)"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def _lib_device_info(local):
    from coevonet_b200 import _lib
    return _lib.device_info(local)


class _NoComm:
    """A single-rank view inside a multi-rank job (the reference run of _sharded_equals_single)."""
    enabled, rank, world, group = False, 0, 1, None

    def all_gather_rows(self, local, shard):
        return local

    def all_reduce_sum(self, t):
        return t

    def all_reduce_max(self, t):
        return t

    def broadcast0(self, t):
        return t


def _sharded_equals_single(engine, layout, FCNetwork, args, dev, comm, rank):
    """One generation of the GLOBAL population, sharded over the ranks, against the same generation run by
    rank 0 alone (evolutionary_strategy.py:236-265): member rewards must be bit-identical (Philox counters use
    global member ids, every rank runs the K1 variant chosen for the global shape); the all-reduced delta may
    differ from the single-rank sum by fp32 summation order only."""
    import torch
    import torch.distributed as dist
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    sh = engine.ESEngine(args, dev, theta, comm=comm)
    sh.evaluate()
    sh.update()
    rewards = torch.stack([comm.all_gather_rows(sh.rewards[r], sh.shard) for r in ROLES])
    delta = sh.delta_cat.clone()
    res = None
    if rank == 0:
        single = engine.ESEngine(args, dev, theta, comm=_NoComm())
        single.evaluate()
        single.update()
        r1 = torch.stack([single.rewards[r] for r in ROLES])
        scale = float(single.delta_cat.abs().max())
        diff = float((single.delta_cat - delta).abs().max())
        same = bool(torch.equal(r1, rewards))
        res = {"equal": bool(same and diff <= 1e-5 * scale), "rewards_bit_identical": same,
               "members_compared": int(r1.numel()), "delta_max_abs_diff": diff, "delta_scale": scale,
               "generations": 1, "k1_variant": int(sh.variant),
               "note": "rank 0 re-runs the whole global population alone; delta differs by the summation order of "
                       "the all-reduce only"}
        del single
    del sh
    torch.cuda.empty_cache()
    dist.barrier()
    return res


def dump_outputs(eng, out_dir):
    """Write what the engine's last generation hands its caller to ``out_dir/<name>.npy``, so that two
    builds run with the same arguments can be compared output for output: per role the members' rewards
    (fp64, this rank's members), the fitness the update used (fp64, all members), the updated base row and
    the update applied to it (fp32, the row's parameters without the pitch padding), and the three rewards
    of the evaluation games (fp64).  About 3.4 MB at the bench workload."""
    import numpy as np
    from coevonet_b200 import layout
    arrays = {"eval_rewards": np.array(eng.last_eval(), dtype=np.float64)}
    for r in ROLES:
        d = layout.fc_dim(layout.OBS_DIM[r])
        arrays[f"rewards_{r}"] = eng.rewards[r].cpu().numpy()
        arrays[f"fitness_{r}"] = eng.fitness[r].cpu().numpy()
        arrays[f"theta_{r}"] = eng.theta[r][:d].cpu().numpy()
        arrays[f"delta_{r}"] = eng.last_delta[r][:d].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        if a.dtype not in (np.float32, np.float64):
            raise TypeError(f"{name}: {a.dtype} is neither float32 nor float64")
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_gpu_arm(ns):
    import numpy as np
    import torch
    import torch.distributed as dist

    from coevonet_b200 import engine, layout, ops
    from coevonet_b200.MPE.fcnetwork import FCNetwork

    # stdout carries exactly one JSON line: keep NCCL's banner ("NCCL version ...") off it
    os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != ns.gpus:
        if world == 1 and ns.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    comm = engine.Comm()

    P = P_PER_GPU * world
    args = _args_bag(P)
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    eng = engine.ESEngine(args, dev, theta, comm=comm)
    n_local = eng.shard.n_local

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (`value`) --------------------------------
    for _ in range(ns.warmup):
        eng.step(sync=False)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(ns.steps):
        eng.step(sync=False)
    e1.record()
    barrier()
    eng.check_status()
    clocks = sampler.stop() if rank == 0 else None
    launches = ops.launch_count - launches0
    ms_total = e0.elapsed_time(e1)
    # the passes below keep stepping the engine: its outputs are those of the last timed step only here
    if ns.dump_outputs and rank == 0:
        dump_outputs(eng, ns.dump_outputs)

    # ---- per-kernel durations for the roofline: the same generation with the three roles back to back
    # on one stream (in the timed region above they overlap on three streams, which is faster but makes
    # a single kernel's duration unobservable) and CUDA events around every K1 call and every member /
    # opponent kernel launch, on the launch stream ------------------------------------------------
    k1_variant, k1_launches = ops.rollout_plan(local, n_local, 1, ENVS, CYCLES)
    ops.kernel_timing_enable(local, True)
    eng.k1_events = []
    roof_steps = max(1, min(ns.steps, 3))
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    r0.record()
    for _ in range(roof_steps):
        eng.step(sync=False)
    r1.record()
    barrier()
    ms_serial = r0.elapsed_time(r1)
    k1_ms = [a.elapsed_time(b) for a, b in eng.k1_events]
    eng.k1_events = None
    member_ms, member_n = ops.kernel_timing_read(local, 0)
    opp_ms, opp_n = ops.kernel_timing_read(local, 1)
    ops.kernel_timing_enable(local, False)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    steps_per_gen = (P * ENVS * 3 + engine.N_EVAL_GAMES) * CYCLES
    value = steps_per_gen * ns.steps / (ms_total * 1e-3)

    # ---- end to end through the host-buffer API (`e2e`) --------------------------
    # inputs of a generation live in pinned host memory (base rows + initial env states, as the
    # reference's host-side env would supply them); results (fitness, updated rows) are read back
    init_host = {r: torch.empty((n_local, 1, ENVS, 11), dtype=torch.float64).pin_memory() for r in ROLES}
    gen_states = ops.init_states(1870300, 0x7000, n_local * ENVS * 3, dev).reshape(3, n_local, 1, ENVS, 11).cpu()
    for i, r in enumerate(ROLES):
        init_host[r].copy_(gen_states[i])
    theta_host = {r: eng.theta[r].cpu().pin_memory() for r in ROLES}
    fit_host = {r: torch.empty(n_local, dtype=torch.float64).pin_memory() for r in ROLES}

    def e2e_step():
        for r in ROLES:
            eng.theta[r].copy_(theta_host[r], non_blocking=True)
        init_dev = {r: init_host[r].to(dev, non_blocking=True) for r in ROLES}
        eng.step(init_by_role=init_dev, sync=False)
        for r in ROLES:
            fit_host[r].copy_(eng.rewards[r], non_blocking=True)
            theta_host[r].copy_(eng.theta[r], non_blocking=True)
        torch.cuda.synchronize()          # the caller holds the generation's results on the host

    h2d = sum(init_host[r].numel() * 8 + theta_host[r].numel() * 4 for r in ROLES)
    d2h = sum(fit_host[r].numel() * 8 + theta_host[r].numel() * 4 for r in ROLES)
    e2e_steps = ns.steps                  # the full --steps, host clock (VERDICT r1 #12)
    for _ in range(min(ns.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = steps_per_gen * e2e_steps / (float(t.item()) * 1e-3)

    # ---- N > 1: the sharded run against a single-rank run of the same GLOBAL population ----------
    sharded = None
    if world > 1:
        sharded = _sharded_equals_single(engine, layout, FCNetwork, args, dev, comm, rank)

    # ---- secondary configs / kernels (bench_secondary.py) -------------------------------------
    secondary = None
    if not ns.no_secondary:
        import bench_secondary as bs
        peaks_s, peaks_src_s = _measured_peaks()
        torch.cuda.empty_cache()
        secondary = {}
        if world == 1:
            secondary["kernels"] = bs.kernel_rooflines(dev, float(peaks_s["hbm_gbs"]), peaks_src_s)
            secondary["config4_dqn_forward"] = bs.config4_dqn_forward(
                dev, float(peaks_s["hbm_gbs"]),
                float(peaks_s.get("bf16_tflops_sustained", peaks_s["bf16_tflops"])) / 2.0)
            torch.cuda.empty_cache()
        secondary["config3_ga"] = bs.config3_ga(dev, comm)
        torch.cuda.empty_cache()
        secondary["config5_dqn_es"] = bs.config5_dqn_es(dev, comm)
        torch.cuda.empty_cache()

    if rank == 0:
        peaks, peaks_src = _measured_peaks()
        fp32_peak = max(ops.fp32_peak(dev, 0), ops.fp32_peak(dev, 1))
        n_sm, _ = _lib_device_info(local)
        sm_max = (clocks or {}).get("sm_max_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        fp32_theory = n_sm * 128 * 2 * sm_max * 1e6 / 1e12          # 128 FMA lanes per SM per clock
        k1_avg_ms = float(np.mean(k1_ms))
        k1_flop = n_local * ENVS * CYCLES * FLOP_PER_WORLD_STEP
        traffic = _k1_traffic()
        hbm_peak = float(peaks["hbm_gbs"])
        # the opponent kernel is timed inside a long step: sustained figure (burst when it is absent)
        tf32_peak = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])) / 2.0
        k1_block = {"k1_variant": {1: "generic", 2: "cluster", 3: "lockstep"}[k1_variant],
                    "k1_kernels_per_call": k1_launches, "k1_ms_per_call": k1_avg_ms, "k1_calls_timed": len(k1_ms),
                    "k1_share_of_step": sum(k1_ms) / ms_serial,
                    "serial_ms_per_step": ms_serial / roof_steps,
                    "timing_note": "kernel durations come from a separate pass with the roles and the kernels of a world "
                                   "step back to back on one stream, every kernel ALONE on all SMs; in the timed region "
                                   "(`value`) the member kernel runs on a share of the SMs beside the opponent kernel",
                    "k1_algorithmic_tflops": k1_flop / (k1_avg_ms * 1e-3) / 1e12,
                    "k1_algorithmic_flop_per_call": k1_flop,
                    "fp32_peak_tflops": fp32_peak,
                    "fp32_peak_source": "FP32 FMA-pipe peak measured live by cev_fp32_peak (MEASURED_PEAKS.json "
                                        "has no FP32 figure)",
                    "fp32_peak_theoretical_tflops": fp32_theory,
                    "fp32_peak_theoretical_def": f"{n_sm} SMs x 128 FMA lanes x 2 x {sm_max:.0f} MHz"}
        if k1_variant == 3 and member_n > 0:
            # dominant kernel: ls_member_tc_kernel, one launch per role and world step; it streams every member row
            # once per launch (algorithmic bytes = rows x D x 4, D averaged over the three roles' launches)
            row_bytes = 4.0 * sum(layout.fc_dim(layout.OBS_DIM[r]) for r in ROLES) / 3.0
            member_us = member_ms / member_n * 1e3
            opp_us = opp_ms / max(opp_n, 1) * 1e3
            alg_bytes = n_local * row_bytes
            achieved = alg_bytes / (member_us * 1e-6) / 1e9
            opp_flop = 2.0 * n_local * ENVS * 2 * 512 * 256          # fc2 of the two opponent seats
            member_fc2_flop = n_local * ENVS * 2 * 512 * 256
            hbm_floor_us = alg_bytes / (hbm_peak * 1e9) * 1e6
            # tensor-pipe floor of the member kernel: 16 k-tiles x 16 tcgen05.mma per member, each occupying the
            # pipe ~45 cycles whatever N <= 64 is (scripts/probe/mma_probe.cu), members spread over all SMs
            mma_floor_us = -(-n_local // n_sm) * 16 * 16 * 45.0 / sm_max
            step_ms = ms_total / ns.steps
            # HBM bytes one generation must move: every member row once per world step (rollouts), written once
            # (K5) and read once more (K6)
            gen_bytes = 3 * alg_bytes * (CYCLES + 2)
            roof = {"kernel": "ls_member_tc_kernel (K1 lockstep, member forward on tcgen05 with the member's own fc2 "
                              "matrix as the M-side operand; one launch per role and world step)",
                    "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved / hbm_peak,
                    "floors": {
                        "per_launch_hbm_us": hbm_floor_us, "per_launch_tensor_us": mma_floor_us,
                        "per_rollout_hbm_bytes_streamed": alg_bytes * CYCLES,
                        "per_rollout_hbm_bytes_if_rows_stayed_on_chip": alg_bytes,
                        "note": "the lockstep form re-streams every member row once per world step (25x the "
                                "once-per-rollout bytes of SURVEY.md 8d): that is a design choice, not the "
                                "algorithm (1.7 GB of member rows per GPU do not fit on chip).  Per launch the HBM "
                                "floor is above the tensor-pipe floor (a tcgen05.mma with N = 32 still occupies the "
                                "pipe ~45 cycles), so `bound` is hbm.  `frac` is the kernel ALONE on all SMs; in "
                                "the timed region it gets a share of the SMs and the opponent kernel the rest, "
                                "see whole_step."},
                    "whole_step": {
                        "hbm_bytes_per_generation": gen_bytes,
                        "achieved_gbs": gen_bytes / (step_ms * 1e-3) / 1e9,
                        "frac_of_hbm_peak": gen_bytes / (step_ms * 1e-3) / 1e9 / hbm_peak,
                        "note": "all HBM traffic a generation needs (rollout streams + K5 write + K6 read) over the "
                                "whole generation time: the rollout streams run under the opponents' MMAs"},
                    "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks_src})",
                    "us_per_launch": member_us, "launches_timed": member_n,
                    "share_of_step": member_ms / ms_serial,
                    "algorithmic_bytes_per_launch": alg_bytes,
                    "algorithmic_bytes_per_unit": row_bytes, "unit_def": "member row per world step",
                    "issued_tf32_tflops": 4 * member_fc2_flop / (member_us * 1e-6) / 1e12,
                    "traffic": traffic["dram_bytes_per_launch"] * n_local / traffic["members"] if traffic else None,
                    "traffic_source": traffic["source"] if traffic else None,
                    "second_kernel": {
                        "kernel": "ls_opp_kernel (tcgen05 kind::tf32, 3 MMAs per product = 3xTF32)",
                        "bound": "tensor", "us_per_launch": opp_us, "launches_timed": opp_n,
                        "share_of_step": opp_ms / ms_serial,
                        "achieved": opp_flop / (opp_us * 1e-6) / 1e12, "unit": "TFLOP/s",
                        "issued_tf32_tflops": 3 * opp_flop / (opp_us * 1e-6) / 1e12,
                        "peak": tf32_peak, "frac": 3 * opp_flop / (opp_us * 1e-6) / 1e12 / tf32_peak,
                        "peak_source": f"half of MEASURED_PEAKS.json bf16_tflops_sustained ({peaks_src}): dense TF32 "
                                       "runs at half the bf16 rate; frac counts the 3 issued MMAs per algorithmic "
                                       "product; alone on 148 SMs the 256 jobs of this shape make 2 rounds (0.86 "
                                       "occupancy), in the timed region the kernel runs on its share of the SMs"}}
        else:
            achieved = k1_flop / (k1_avg_ms * 1e-3) / 1e12
            roof = {"kernel": "rollout_cluster_kernel<16> (K1)", "bound": "fp32", "achieved": achieved,
                    "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                    "traffic": None}
        roof.update(k1_block)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": ns.steps,
            "warmup": ns.warmup, "ms_per_step": ms_total / ns.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(world),
            "agent_steps_per_sec": 3 * value,
            "roofline": roof,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps},
            "gpu_launches": launches,
            "clocks": clocks,
        }
        if sharded is not None:
            line["sharded_equals_single"] = sharded["equal"]
            line["sharded_check"] = sharded
        if secondary is not None:
            line["secondary"] = secondary
        if world == 1 and not ns.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_block()
            line["parity"] = parity_block(dev)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-secondary", dest="no_secondary", action="store_true",
                    help="skip the secondary configs / per-kernel rooflines (bench_secondary.py)")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs to DIR/<name>.npy (rank 0)")
    ns = ap.parse_args()
    if ns.steps < 1 or ns.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if ns.impl == "reference" and ns.dump_outputs:
        ap.error("--dump-outputs writes the outputs of this build's GPU path (--impl b200)")
    if ns.impl == "reference":
        return run_reference_arm(ns)
    return run_gpu_arm(ns)


if __name__ == "__main__":
    sys.exit(main())
