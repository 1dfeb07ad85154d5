"""Device times of the separable-NES kernels (diag K5 / K6 / apply) next to the isotropic forms, and of one ES
generation at the bench shape with the defaults and with separable NES + mirrored sampling + centered ranks.  CUDA
events around repeated launches after warm-up; the forms of a kernel are timed alternately in the same process
(helpers of scripts/time_es_options.py).  Writes <out-dir>/r04_snes.json.

    python scripts/time_snes.py --out-dir OUT
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from coevonet_b200 import engine, layout, ops  # noqa: E402
from time_es_options import HBM_TBPS, REPS, alternate, card  # noqa: E402

ROLES = layout.ROLES


def _sigma_row(in_dim, value):
    row = torch.zeros(layout.fc_pitch(in_dim))
    row[torch.from_numpy(layout.fc_perturbable_index(in_dim))] = value
    return row.cuda()


def k5(rows):
    pitch = layout.fc_pitch(10)
    theta = torch.randn(pitch, device="cuda") * 0.05
    sigma = _sigma_row(10, 0.05)
    out = torch.empty((rows, pitch), device="cuda")
    r = alternate({
        "plain": lambda: ops.es_perturb(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out),
        "diag": lambda: ops.es_perturb_diag(theta, sigma, 10, 1, "agent_0", 0, 0, rows, out=out),
        "mirrored": lambda: ops.es_perturb_mirrored(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out),
        "diag_mirrored": lambda: ops.es_perturb_diag(theta, sigma, 10, 1, "agent_0", 0, 0, rows, mirrored=True,
                                                     out=out)},
        20 if rows <= 1024 else 5)
    floor_us = rows * pitch * 4 / (HBM_TBPS * 1e12) * 1e6
    for v in r.values():
        v["fraction_of_hbm_write_floor"] = round(floor_us / v["us"], 3)
    return {"rows": rows, "bytes_written": rows * pitch * 4, "hbm_write_floor_us": round(floor_us, 1), **r}


def k6(rows):
    pitch = layout.fc_pitch(10)
    fit = torch.randn(rows, dtype=torch.float64, device="cuda")
    theta = torch.randn(pitch, device="cuda") * 0.05
    members = ops.es_perturb(theta, 10, 0.05, 1, "agent_0", 0, 0, rows)
    g_mu, g_sigma = torch.empty(pitch, device="cuda"), torch.empty(pitch, device="cuda")
    return {"rows": rows, **alternate({
        "regenerated": lambda: ops.es_update(fit, 10, 0.05, 0.1, rows, 1, "agent_0", 0, 0),
        "diag": lambda: ops.es_update_diag(fit, 10, rows, 1, "agent_0", 0, 0, g_mu=g_mu, g_sigma=g_sigma),
        "regenerated_mirrored": lambda: ops.es_update_mirrored(fit, 10, 0.05, 0.1, rows, 1, "agent_0", 0, 0),
        "diag_mirrored": lambda: ops.es_update_diag(fit, 10, rows, 1, "agent_0", 0, 0, mirrored=True, g_mu=g_mu,
                                                    g_sigma=g_sigma),
        "members": lambda: ops.es_update_members(fit, members, theta, 10, 0.05, 0.1, rows)},
        20 if rows <= 1024 else 5)}


def apply():
    in_dims = [layout.OBS_DIM[r] for r in ROLES]
    n = sum(layout.fc_pitch(d) for d in in_dims)
    theta = torch.randn(n, device="cuda")
    sigma = torch.cat([_sigma_row(d, 0.05) for d in in_dims])
    g_mu, g_sigma = torch.randn(n, device="cuda") * 1e-3, torch.randn(n, device="cuda") * 1e-3
    r = alternate({"diag": lambda: ops.es_apply_diag(theta, sigma, g_mu, g_sigma, in_dims, lr=1e-3,
                                                     sigma_lr=[0.008, 0.008, 0.008], sigma_min=0.001, sigma_max=0.2),
                   "axpy": lambda: ops.axpy(1.0, g_mu, theta)}, 20)
    return {"floats": n, **r}


def generation():
    import bench
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    on = dict(es_distribution="separable", mirrored_sampling=True, fitness_shaping="centered_rank", learning_rate=1.0)
    engs = {}
    for name, opts in (("defaults", {}), ("separable_mirrored_ranks", on)):
        args = bench._args_bag(bench.P_PER_GPU)
        for k, v in opts.items():
            setattr(args, k, v)
        engs[name] = engine.ESEngine(args, torch.device("cuda", torch.cuda.current_device()), theta)
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 10)
    for e in engs.values():
        e.check_status()
    out = {"population": bench.P_PER_GPU, "envs_per_member": bench.ENVS, "roles": 3}
    for k, v in res.items():
        out[k] = {"ms_per_generation": round(v["us"] / 1e3, 3), "ms_all": [round(x / 1e3, 3) for x in v["us_all"]]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    method = (f"CUDA events, 3 warm-up calls, a device sleep queued ahead of each window, median of {REPS} windows, "
              f"forms alternated; HBM floor = bytes / {HBM_TBPS} TB/s (data sheet)")
    res = {"card": card(), "method": method, "k5": [k5(1024), k5(8192)], "k6": [k6(1024), k6(8192)],
           "apply": apply(), "generation": generation()}
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r04_snes.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
