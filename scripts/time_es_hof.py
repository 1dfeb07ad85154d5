"""Device time of one Co-ES generation at the bench shape (1,024 members, 3 roles) with and without the Hall of Fame:
the defaults at E = 16, K = 4 opponent sets at E = 4 (the same 16 games per member) and K = 4 at E = 16.  The three
engines step alternately in the same process, medians of the windows (helpers of scripts/time_es_options.py).  A
separate profiled pass splits a generation into its kernels, so the cost of each extra opponent set (the opponent
fc2 split, ls_split_w2_kernel, and the opponent forward) is visible.  Also the draw + gather of the opponents.
Writes <out-dir>/r05_es_hof.json.

    python scripts/time_es_hof.py --out-dir OUT
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
from time_es_options import REPS, alternate, card  # noqa: E402

ROLES = layout.ROLES
FORMS = {"default_E16": dict(envs_per_member=16),
         "hof_K4_E4": dict(envs_per_member=4, es_hof_size=8, es_hof_opponents=4),
         "hof_K4_E16": dict(envs_per_member=16, es_hof_size=8, es_hof_opponents=4)}
PROFILED_GENERATIONS = 3


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
        for _ in range(8):                               # fill the archive: every draw then has 8 slots to pick from
            engs[name].step(sync=False)
    torch.cuda.synchronize()
    return engs


def generation(engs):
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 10)
    for e in engs.values():
        e.check_status()
    out = {}
    for k, v in res.items():
        e = engs[k]
        out[k] = {"K": e.K, "E": e.E, "games_per_member": e.K * e.E, "variant": e.variant,
                  "ms_per_generation": round(v["us"] / 1e3, 3), "ms_all": [round(x / 1e3, 3) for x in v["us_all"]]}
    return out


def kernels(engs):
    """Device microseconds per generation of every kernel (torch.profiler, a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, e in engs.items():
        e.step(sync=False)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(PROFILED_GENERATIONS):
                e.step(sync=False)
            torch.cuda.synchronize()
        rows = {}
        for ev in prof.key_averages():
            t = getattr(ev, "device_time_total", None)
            if t is None:
                t = getattr(ev, "cuda_time_total", 0.0)
            if t > 0:
                rows[ev.key] = {"us_per_generation": round(t / PROFILED_GENERATIONS, 1),
                                "launches_per_generation": ev.count / PROFILED_GENERATIONS}
        out[name] = dict(sorted(rows.items(), key=lambda kv: -kv[1]["us_per_generation"]))
    return out


def hof_ops(engs):
    e = engs["hof_K4_E16"]
    newest = (e.hof_head - 1) % e.hof_size
    return alternate({"draw": lambda: ops.es_hof_opponents(e.seed, 3, 4, 8, newest, e.device, out=e.hof_ids),
                      "gather": lambda: ops.gather_rows(e.hof_ring, e.hof_ids, out=e.hof_opp)}, 50)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    res = {"card": card(),
           "method": f"CUDA events around 10 generations per window, a device sleep queued ahead of each window, "
                     f"median of {REPS} windows, the three engines alternated window by window; kernel split from "
                     f"torch.profiler over {PROFILED_GENERATIONS} generations per engine in a separate pass",
           "population": 1024, "roles": 3}
    engs = _engines()
    res["generation"] = generation(engs)
    res["hof_ops_us"] = hof_ops(engs)
    res["kernels"] = kernels(engs)
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r05_es_hof.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("card", "generation", "hof_ops_us", "card_after")}, indent=1))
    for name, rows in res["kernels"].items():
        print(name)
        for k, v in list(rows.items())[:8]:
            print(f"   {v['us_per_generation']:10.1f} us  x{v['launches_per_generation']:g}  {k[:90]}")


if __name__ == "__main__":
    main()
