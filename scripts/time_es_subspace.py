"""Device times of Co-ES guided search: the subspace K5 next to the isotropic K5 (plain and mirrored, 1,024 and 8,192
rows, k = 4, 16, 32 with a full basis), the basis kernel chain for the three roles, and one ES generation at the bench
shape with the defaults and with --es_subspace_dim 16.  CUDA events around repeated launches after warm-up; the
forms are timed alternately in the same process (helpers of scripts/time_es_options.py).  Writes
<out-dir>/r06_es_subspace.json.

    python scripts/time_es_subspace.py --out-dir OUT
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
DIMS = (4, 16, 32)
IN_DIMS = [layout.OBS_DIM[r] for r in ROLES]


def _full_basis(k):
    """A ring of k random estimates on the Linear entries of the three roles and its basis (k_eff = k per role)."""
    n = sum(layout.fc_pitch(d) for d in IN_DIMS)
    mask = torch.zeros(n, dtype=torch.bool)
    off = 0
    for d in IN_DIMS:
        mask[off + torch.from_numpy(layout.fc_perturbable_index(d))] = True
        off += layout.fc_pitch(d)
    g = torch.Generator().manual_seed(k)
    ring = (torch.randn((k, n), generator=g) * mask).cuda()
    U, ke = ops.es_subspace_basis(ring, k - 1, k, IN_DIMS)
    assert ke.tolist() == [k] * 3
    return ring, U, ke


def k5(rows):
    pitch = layout.fc_pitch(10)                      # agent_0, the first role of the concatenated rows
    theta = torch.randn(pitch, device="cuda") * 0.05
    out = torch.empty((rows, pitch), device="cuda")
    fns = {"k5": lambda: ops.es_perturb(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out),
           "k5_mirrored": lambda: ops.es_perturb_mirrored(theta, 10, 0.05, 1, "agent_0", 0, 0, rows, out=out)}
    keep = []
    for k in DIMS:
        _, U, ke = _full_basis(k)
        keep.append(U)
        Ur, kr = U[:, :pitch], ke[0:1]
        for mirrored in (False, True):
            fns[f"subspace_k{k}" + ("_mirrored" if mirrored else "")] = (
                lambda Ur=Ur, kr=kr, m=mirrored: ops.es_perturb_subspace(theta, 10, 0.05, Ur, kr, 0.5, 1, "agent_0", 0,
                                                                         0, rows, mirrored=m, out=out))
    r = alternate(fns, 20 if rows <= 1024 else 5)
    floor_us = rows * pitch * 4 / (HBM_TBPS * 1e12) * 1e6
    for v in r.values():
        v["fraction_of_hbm_write_floor"] = round(floor_us / v["us"], 3)
    for k in DIMS:
        for sfx in ("", "_mirrored"):
            r[f"subspace_k{k}{sfx}"]["ratio_to_k5"] = round(r[f"subspace_k{k}{sfx}"]["us"] / r["k5" + sfx]["us"], 3)
    return {"rows": rows, "bytes_written": rows * pitch * 4, "hbm_write_floor_us": round(floor_us, 1), **r}


def basis():
    fns = {}
    for k in DIMS:
        ring, U, ke = _full_basis(k)
        fns[f"k{k}"] = lambda ring=ring, U=U, ke=ke, k=k: ops.es_subspace_basis(ring, k - 1, k, IN_DIMS, out=U, k_eff=ke)
    return {"roles": 3, "kernels_per_call": 6, **alternate(fns, 20)}


def generation():
    import bench
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    engs = {}
    for name, opts in (("defaults", {}), ("subspace_k16", dict(es_subspace_dim=16))):
        args = bench._args_bag(bench.P_PER_GPU)
        for k, v in opts.items():
            setattr(args, k, v)
        engs[name] = engine.ESEngine(args, torch.device("cuda", torch.cuda.current_device()), theta)
        for _ in range(18):                              # fill the ring: k_eff = 16 from here on
            engs[name].step(sync=False)
    torch.cuda.synchronize()
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 10)
    for e in engs.values():
        e.check_status()
    out = {"population": bench.P_PER_GPU, "envs_per_member": bench.ENVS, "roles": 3,
           "subspace_rank": engs["subspace_k16"].subspace_keff.cpu().tolist()}
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
              f"forms alternated; HBM floor = bytes / {HBM_TBPS} TB/s (data sheet); generations: 10 per window after "
              f"18 warm-up generations that fill the estimate ring")
    res = {"card": card(), "method": method, "k5": [k5(1024), k5(8192)], "basis": basis(),
           "generation": generation()}
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r06_es_subspace.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
