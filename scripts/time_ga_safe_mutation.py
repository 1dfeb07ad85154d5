"""Device time of the Co-GA safe mutations: K3 plain against K3 with scale rows at 1,024 and 8,192 child rows (the
forms alternated, against the HBM write floor of the rows); the scale chain (cev_ga_safe_scale_f32) per role at
E = 2, 16 and 64; one GA generation at 8,192 members on one GPU with the BASELINE configs[2] settings (hof 3,
5 elites, adaptive, fitness sharing), the default engine against --ga_safe_mutation, alternated window by window
(helpers of scripts/time_es_options.py); and the largest errors of the kernel's sensitivity against the fp64 oracle
(relative to the tests' tolerance).  Writes <out-dir>/r09_ga_safe_mutation.json.

    python scripts/time_ga_safe_mutation.py --out-dir OUT
"""
import argparse
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from coevonet_b200 import _lib, engine, layout, ops  # noqa: E402
from oracle import ga_safe_mutation as gsm, layout as olayout  # noqa: E402
from time_es_options import HBM_TBPS, REPS, alternate, card  # noqa: E402

ROLES = layout.ROLES
FORMS = {"default": {}, "safe_mutation": dict(ga_safe_mutation=True)}


def _obs(role):
    return ops.novelty_probe_obs(ops.init_states(11, engine.NOVELTY_PROBE_TAG, _lib.NOVELTY_PROBES, "cuda"), role)


def _elites(role, E):
    in_dim = layout.OBS_DIM[role]
    base = ops.fc_init(in_dim, 11, role, 0, 1, "cuda")
    return ops.ga_repopulate(base, layout.fc_dim(in_dim), 0.05, 11, role, 0, 1, E)


def k3(rows):
    role, in_dim = "agent_0", 10
    elites = _elites(role, 5)
    scale = ops.ga_safe_scale(elites, in_dim, _obs(role), 0.01)
    out = torch.empty((rows, elites.shape[1]), device="cuda")
    D = layout.fc_dim(in_dim)
    r = alternate({"plain": lambda: ops.ga_repopulate(elites, D, 0.05, 1, role, 0, 0, rows, out=out),
                   "safe": lambda: ops.ga_repopulate(elites, D, 0.05, 1, role, 0, 0, rows, out=out, scale=scale)},
                  20 if rows <= 1024 else 5)
    floor_us = rows * elites.shape[1] * 4 / (HBM_TBPS * 1e12) * 1e6
    for v in r.values():
        v["fraction_of_hbm_write_floor"] = round(floor_us / v["us"], 3)
    return {"rows": rows, "bytes_written": rows * elites.shape[1] * 4, "hbm_write_floor_us": round(floor_us, 1), **r}


def chain(E):
    out = {"E": E}
    for role in ("agent_0", "adversary_0"):
        in_dim = layout.OBS_DIM[role]
        elites, obs = _elites(role, E), _obs(role)
        scale = torch.empty_like(elites)
        r = alternate({role: lambda: ops.ga_safe_scale(elites, in_dim, obs, 0.01, out=scale)}, 20)[role]
        out[f"in_dim_{in_dim}"] = r
    return out


def errors():
    """Largest |s_gpu - s_ref| / (1e-4 s_ref + 1e-5 magnitude) and largest relative error of s, over fc_init rows,
    sigma-0.05 mutants and rows with LN gamma x40 / x0.02 and fc2 x250 / x0.01, parents with mask margin > 1e-5 (as
    in tests/test_gpu_ga_safe_mutation.py)."""
    res = {}
    for role in ("agent_0", "adversary_0"):
        in_dim = layout.OBS_DIM[role]
        D = layout.fc_dim(in_dim)
        obs = _obs(role)
        base = ops.fc_init(in_dim, 11, role, 0, 2, "cuda")
        rows = [base, ops.ga_repopulate(base, D, 0.05, 11, role, 1, 1, 2)]
        segs = {name: (off, int(np.prod(shape))) for name, off, shape, _ in olayout.fc_segments(in_dim)[0]}
        for name, f in (("ln1.weight", 40.0), ("ln1.weight", 0.02), ("fc2.weight", 250.0), ("fc2.weight", 0.01)):
            row = base[0:1].clone()
            off, n = segs[name]
            row[0, off:off + n] *= f
            rows.append(row)
        rows = torch.cat(rows).contiguous()
        c = ops.ga_safe_scale(rows, in_dim, obs, 1e-30).cpu().numpy().astype(np.float64)
        names = ["fc_init 0", "fc_init 1", "mutant 1", "mutant 2", "ln1.weight x40", "ln1.weight x0.02",
                 "fc2.weight x250", "fc2.weight x0.01"]
        per = []
        for e, row in enumerate(rows.cpu().numpy()):
            s_ref, mag, margin = gsm.sensitivity(row[:D], in_dim, obs.cpu().numpy())
            nz = c[e, :D] != 1.0
            err = np.abs(1.0 / c[e, :D][nz] - s_ref[nz])
            ratio = err / (1e-4 * s_ref[nz] + 1e-5 * mag[nz])
            per.append({"parent": names[e], "mask_margin": float(margin), "compared": bool(margin > 1e-5),
                        "max_error_over_tolerance": float(ratio.max()),
                        "entries_over_tolerance": int((ratio > 1).sum()),
                        "max_relative_error": float((err / s_ref[nz]).max())})
        cmp = [p for p in per if p["compared"]]
        res[f"in_dim_{in_dim}"] = {"parents": per, "parents_with_margin": len(cmp),
                                   "max_error_over_tolerance": max(p["max_error_over_tolerance"] for p in cmp),
                                   "max_relative_error": max(p["max_relative_error"] for p in cmp)}
    return res


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(),
           "method": f"CUDA events around n back-to-back calls (20 or 5 kernels / chains, 5 generations) per window "
                     f"after warm-up, a device sleep queued ahead of each window, median of {REPS} windows, forms "
                     f"alternated window by window; HBM write floor = rows x pitch x 4 B / {HBM_TBPS} TB/s",
           "k3": [k3(1024), k3(8192)],
           "scale_chain": [chain(2), chain(16), chain(64)],
           "sensitivity_errors": errors()}
    torch.cuda.empty_cache()
    res["generation"] = {"population": 8192, "n_gpus": 1, "hof_size": 3, "elites": 5, **generation(_engines())}
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r09_ga_safe_mutation.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
