"""Device time of the Co-GA novelty search: the population + archive k-NN kernel at (members, population) =
(1,024, 1,024), (8,192, 8,192) and (8,192, 65,536) with an archive of 1,024 filled entries and k = 10, against its
issue floor (2 FP32 lane operations per term over 148 SMs x 128 lanes per clock at the card's maximum SM clock); one
GA generation at 8,192 members on one GPU with the BASELINE configs[2] settings (hof 3, 5 elites, adaptive, fitness
sharing) with --ga_novelty_weight 0 and 0.5, the engines alternated window by window (helpers of
scripts/time_es_options.py); and a torch.profiler split of the novelty generation in a separate pass.  Writes
<out-dir>/r08_ga_novelty.json.

    python scripts/time_ga_novelty.py --out-dir OUT
"""
import argparse
import json
import os
import re
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from coevonet_b200 import _lib, engine, layout, ops  # noqa: E402
from time_es_hof import kernels  # noqa: E402
from time_es_options import REPS, alternate, card  # noqa: E402

ROLES = layout.ROLES
FORMS = {"default": {}, "novelty_w05": dict(ga_novelty_weight=0.5)}
#: kernel names of the profiled split, by the part of the novelty search they belong to
PARTS = {"characterisation": ("novelty_bc_kernel",), "all_gather": ("nccl", "AllGather", "Memcpy", "cat"),
         "knn": ("ga_novelty_knn_kernel", "ga_novelty_merge_kernel"), "ranks": ("centered_ranks",)}


def _max_sm_clock_ghz():
    m = re.search(r"(\d+)\s*MHz\s*$", card()["nvidia_smi"])
    return int(m.group(1)) / 1e3 if m else None


def knn_kernel(n, P, filled=1024, k=10):
    """The k-NN of n members (rows 0 .. n-1) against P population rows and `filled` archive entries; the inputs
    are kernel-made characterisations of sigma-0.05 members."""
    in_dim = 10
    obs = ops.novelty_probe_obs(ops.init_states(11, engine.NOVELTY_PROBE_TAG, _lib.NOVELTY_PROBES, "cuda"), "agent_0")
    theta = ops.fc_init(in_dim, 11, "agent_0", 0, 1, "cuda")[0]
    pop = torch.empty((P, _lib.NOVELTY_BC_DIM), device="cuda")
    for a in range(0, P, 8192):
        b = min(P, a + 8192)
        rows = ops.es_perturb(theta, in_dim, 0.05, 11, "agent_0", 0, a, b - a)
        ops.novelty_bc(rows, in_dim, obs, out=pop[a:b])
        del rows
    ring = pop[:filled].flip(0).contiguous() + 1e-3
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    r = alternate({"knn": lambda: ops.ga_novelty_knn(pop[:n], 0, pop, ring, filled, k, out=out)},
                  20 if n * P <= 1 << 20 else 5)["knn"]
    terms = n * (P - 1 + filled) * _lib.NOVELTY_BC_DIM
    ghz = _max_sm_clock_ghz()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    floor_us = 2 * terms / (n_sm * 128 * ghz * 1e9) * 1e6 if ghz else None
    return {"members": n, "population": P, "archive_filled": filled, "k": k, "us": round(r["us"], 1),
            "us_all": r["us_all"], "member_candidate_dimension_terms": terms,
            "issue_floor_us": round(floor_us, 1) if floor_us else None,
            "fraction_of_issue_floor": round(floor_us / r["us"], 3) if floor_us else None,
            "achieved_fp32_tops": round(2 * terms / (r["us"] * 1e-6) / 1e12, 2)}


def _engines(P=8192):
    dev = torch.device("cuda", torch.cuda.current_device())
    engs = {}
    for name, opts in FORMS.items():
        args = types.SimpleNamespace(
            algorithm="GA", generations=100, population=P, hof_size=3, game="simple_adversary_v3",
            mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
            learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=5,
            adaptive=True, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
            early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32",
            save=False, envs_per_member=1, reference_compat=True, init_states="device",
            seed=1870300, plots=False, record_history=False, **opts)
        pop = {r: ops.fc_init(layout.OBS_DIM[r], 7, r, 0, P, dev) for r in ROLES}
        hof = {r: ops.fc_init(layout.OBS_DIM[r], 7, r, P, 3, dev) for r in ROLES}
        founder = {r: ops.fc_init(layout.OBS_DIM[r], 7, r, P - 1, 1, dev)[0] for r in ROLES}
        engs[name] = engine.GAEngine(args, dev, pop, hof, founder)
        for _ in range(3):
            engs[name].step(sync=False)
    torch.cuda.synchronize()
    return engs


def generation(engs):
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 5)
    for e in engs.values():
        e.check_status()
    return {k: {"ms_per_generation": round(v["us"] / 1e3, 3), "ms_all": [round(x / 1e3, 3) for x in v["us_all"]]}
            for k, v in res.items()}


def split(prof_rows):
    """Device microseconds per generation of the novelty search's parts, from the profiled kernel table."""
    out = {p: 0.0 for p in PARTS}
    for name, v in prof_rows.items():
        for p, keys in PARTS.items():
            if any(key in name for key in keys):
                out[p] += v["us_per_generation"]
                break
    return {p: round(v, 1) for p, v in out.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(),
           "method": f"CUDA events around n back-to-back calls (20 or 5 kernels, 5 generations) per window after "
                     f"warm-up, a device sleep queued ahead of each window, median of {REPS} windows, the two engines "
                     f"alternated window by window; issue floor = 2 x terms / (SMs x 128 lanes x max SM clock); "
                     f"kernel split from torch.profiler in a separate pass",
           "knn_kernel": [knn_kernel(1024, 1024), knn_kernel(8192, 8192), knn_kernel(8192, 65536)]}
    torch.cuda.empty_cache()
    engs = _engines()
    res["generation"] = {"population": 8192, "n_gpus": 1, "hof_size": 3, "elites": 5, **generation(engs)}
    prof = kernels({"novelty_w05": engs["novelty_w05"]})["novelty_w05"]
    res["novelty_w05_split_us_per_generation"] = split(prof)
    res["kernels_novelty_w05"] = prof
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r08_ga_novelty.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "kernels_novelty_w05"}, indent=1))
    for k, v in list(res["kernels_novelty_w05"].items())[:14]:
        print(f"   {v['us_per_generation']:10.1f} us  x{v['launches_per_generation']:g}  {k[:90]}")


if __name__ == "__main__":
    main()
