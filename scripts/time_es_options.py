"""Device times of the opt-in Co-ES update kernels (mirrored K5 / K6, centered ranks, fused apply) and of one ES
generation at the bench shape with the options off and on.  CUDA events around repeated launches after warm-up;
the two forms of a kernel are timed alternately in the same process.  Writes <out-dir>/r03_es_options.json.

    python scripts/time_es_options.py --out-dir OUT
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from coevonet_b200 import engine, layout, ops  # noqa: E402

HBM_TBPS = 7.7           # HGX B200 data sheet, one GPU: the write floors below are bytes / this rate
ROLES = layout.ROLES
REPS = 5


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def timed(fn, n):
    """Mean device microseconds of one call over n back-to-back calls (after 3 warm-up calls).  A device sleep is
    queued ahead of the window, so the host has enqueued the n calls before the GPU reaches them: the events time
    the kernels, not the host's enqueue rate (the small kernels here run faster than one Python call)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda._sleep(20_000_000)                       # ~10 ms at 1.965 GHz
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def alternate(fns, n):
    """{name: median over REPS of timed(fn, n)}, the forms interleaved rep by rep."""
    res = {k: [] for k in fns}
    for _ in range(REPS):
        for k, fn in fns.items():
            res[k].append(timed(fn, n))
    return {k: {"us": statistics.median(v), "us_all": [round(x, 2) for x in v]} for k, v in res.items()}


def k5(rows):
    pitch = layout.fc_pitch(10)
    theta = torch.randn(pitch, device="cuda") * 0.05
    out = torch.empty((rows, pitch), device="cuda")
    r = alternate({"plain": lambda: ops.es_perturb(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out),
                   "mirrored": lambda: ops.es_perturb_mirrored(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out)},
                  20 if rows <= 1024 else 5)
    floor_us = rows * pitch * 4 / (HBM_TBPS * 1e12) * 1e6
    for v in r.values():
        v["fraction_of_hbm_write_floor"] = round(floor_us / v["us"], 3)
    return {"rows": rows, "bytes_written": rows * pitch * 4, "hbm_write_floor_us": round(floor_us, 1), **r}


def k6(rows):
    fit = torch.randn(rows, dtype=torch.float64, device="cuda")
    return {"rows": rows, **alternate(
        {"plain": lambda: ops.es_update(fit, 10, 0.05, 0.1, rows, 1, "agent_0", 0, 0),
         "mirrored": lambda: ops.es_update_mirrored(fit, 10, 0.05, 0.1, rows, 1, "agent_0", 0, 0)},
        20 if rows <= 1024 else 5)}


def ranks(P):
    f = torch.round(torch.randn(P, dtype=torch.float64, device="cuda") * 10) / 10
    r = alternate({"centered_ranks": lambda: ops.centered_ranks(f)}, 20 if P <= 8192 else 5)["centered_ranks"]
    r["gcompares_per_s"] = round(P * P / (r["us"] * 1e-6) / 1e9, 1)
    return {"P": P, **r}


def apply():
    in_dims = [layout.OBS_DIM[r] for r in ROLES]
    n = sum(layout.fc_pitch(d) for d in in_dims)
    theta, delta = torch.randn(n, device="cuda"), torch.randn(n, device="cuda") * 1e-3
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    r = alternate({"adam": lambda: ops.es_apply(theta, delta, in_dims, optimizer="adam", lr=1e-3, l2_coeff=0.005,
                                                 t=1, m=m, v=v),
                   "sgd_l2": lambda: ops.es_apply(theta, delta, in_dims, optimizer="sgd", lr=1e-3, l2_coeff=0.005),
                   "axpy": lambda: ops.axpy(1.0, delta, theta)}, 20)
    return {"floats": n, **r}


def generation():
    sys.path.insert(0, ROOT)
    import bench
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    on = dict(mirrored_sampling=True, fitness_shaping="centered_rank", es_optimizer="adam", learning_rate=0.01,
              l2_coeff=0.005)
    engs = {}
    for name, opts in (("defaults", {}), ("all_options", on)):
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
    res = {"card": card(), "method": method,
           "k5": [k5(1024), k5(8192)], "k6_regenerated": [k6(1024), k6(8192)],
           "centered_ranks": [ranks(P) for P in (1024, 8192, 65536)], "apply": apply(), "generation": generation()}
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r03_es_options.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
