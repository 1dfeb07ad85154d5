"""Device time of the Co-ES novelty search: the behaviour-characterisation kernel at 1,024 and 8,192 member rows
against its HBM floor, the k-NN kernel against archives of 1,024 and 4,096 entries, and one generation at the bench
shape (1,024 members x 16 envs x 3 roles) with and without --es_novelty_weight 0.5 --fitness_shaping centered_rank
(and with the ranks alone), the engines alternated window by window (helpers of scripts/time_es_options.py), and a
profiled kernel split of the novelty generation.  Writes <out-dir>/r07_es_novelty.json.  The characterisation's error
against the oracle is measured by tests/tools/novelty_bc_err.py.

    python scripts/time_es_novelty.py --out-dir OUT
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from coevonet_b200 import _lib, engine, layout, ops  # noqa: E402
from time_es_hof import kernels  # noqa: E402
from time_es_options import HBM_TBPS, alternate, card  # noqa: E402

ROLES = layout.ROLES
FORMS = {"default": {}, "ranks": dict(fitness_shaping="centered_rank"),
         "novelty_w05": dict(fitness_shaping="centered_rank", es_novelty_weight=0.5)}


def _members(rows, role="agent_0"):
    in_dim = layout.OBS_DIM[role]
    theta = ops.fc_init(in_dim, 11, role, 0, 1, "cuda")[0]
    return ops.es_perturb(theta, in_dim, 0.05, 11, role, 0, 0, rows)


def _obs(role="agent_0"):
    return ops.novelty_probe_obs(ops.init_states(11, engine.NOVELTY_PROBE_TAG, _lib.NOVELTY_PROBES, "cuda"), role)


def bc_kernel(rows):
    """The characterisation kernel at `rows` members of agent_0 (in_dim 10); every call reads all rows from HBM (the
    rows are larger than L2)."""
    members, obs = _members(rows), _obs()
    out = torch.empty((rows, _lib.NOVELTY_BC_DIM), device="cuda")
    r = alternate({"bc": lambda: ops.novelty_bc(members, 10, obs, out=out)}, 20 if rows <= 1024 else 5)["bc"]
    bytes_read = rows * layout.fc_dim(10) * 4
    floor_us = bytes_read / (HBM_TBPS * 1e12) * 1e6
    flops = rows * 2 * _lib.NOVELTY_PROBES * (10 * layout.H1 + layout.H1 * layout.H2 + layout.H2 * layout.NACT)
    del members
    return {"rows": rows, "bytes_read": bytes_read, "hbm_floor_us": round(floor_us, 1), "us": round(r["us"], 1),
            "us_all": r["us_all"], "fraction_of_hbm_floor": round(floor_us / r["us"], 3),
            "forward_flop": flops, "achieved_tflops": round(flops / (r["us"] * 1e-6) / 1e12, 2)}


def knn_kernel(archive, n=1024, k=10):
    obs = _obs()
    bc = ops.novelty_bc(_members(n), 10, obs)
    ring = ops.novelty_bc(_members(archive + 8)[8:], 10, obs).contiguous()
    out = torch.empty(n, dtype=torch.float64, device="cuda")
    r = alternate({"knn": lambda: ops.novelty_knn(bc, ring, archive, k, out=out)}, 20)["knn"]
    terms = n * archive * _lib.NOVELTY_BC_DIM
    return {"members": n, "archive": archive, "k": k, "us": round(r["us"], 1), "us_all": r["us_all"],
            "member_entry_dimension_terms": terms,
            "fp64_ops": 3 * terms, "achieved_fp64_gops": round(3 * terms / (r["us"] * 1e-6) / 1e9, 1)}


def _engines():
    import bench
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    engs = {}
    for name, opts in FORMS.items():
        args = bench._args_bag(bench.P_PER_GPU)
        for k, v in opts.items():
            setattr(args, k, v)
        engs[name] = engine.ESEngine(args, torch.device("cuda", torch.cuda.current_device()), theta)
        for _ in range(12):                              # the archive then holds more than k = 10 entries
            engs[name].step(sync=False)
    torch.cuda.synchronize()
    return engs


def generation(engs):
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 10)
    for e in engs.values():
        e.check_status()
    return {k: {"E": engs[k].E, "ms_per_generation": round(v["us"] / 1e3, 3),
                "ms_all": [round(x / 1e3, 3) for x in v["us_all"]]} for k, v in res.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(),
           "method": "CUDA events around n back-to-back calls (20 or 5 kernels, 10 generations) per window, a device "
                     "sleep queued ahead of each window, median of 5 windows, forms alternated window by window; "
                     "HBM floor = member bytes read / 7.7 TB/s; kernel split from torch.profiler over 3 generations "
                     "in a separate pass",
           "bc_kernel": [bc_kernel(1024), bc_kernel(8192)],
           "knn_kernel": [knn_kernel(1024), knn_kernel(4096)]}
    engs = _engines()
    res["generation"] = {"population": 1024, "roles": 3, **generation(engs)}
    res["kernels_novelty_w05"] = kernels({"novelty_w05": engs["novelty_w05"]})["novelty_w05"]
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r07_es_novelty.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "kernels_novelty_w05"}, indent=1))
    for k, v in list(res["kernels_novelty_w05"].items())[:12]:
        print(f"   {v['us_per_generation']:10.1f} us  x{v['launches_per_generation']:g}  {k[:90]}")


if __name__ == "__main__":
    main()
