"""Device times of Co-ES LM-MA-ES: per role (agent_0) at 1,024 and 8,192 rows and m = 4, 8, 16, 32 vectors in use,
the projection + coefficients and the LM-MA K5 beside the isotropic K5 and the subspace K5 at the same k; the
recombination (mu = 512 of 1,024) and the apply of the three roles at m = 8; and one ES generation at the bench shape
(BASELINE config 2: 1,024 members x 16 games x 3 roles) with the defaults and with --es_distribution lmma
--es_lmma_memory 8 (all 8 vectors in use).  CUDA events around repeated launches after warm-up; the forms are timed
alternately in the same process (helpers of scripts/time_es_options.py).  Writes <out-dir>/r10_es_lmma.json.

    python scripts/time_es_lmma.py --out-dir OUT
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
from time_es_subspace import _full_basis  # noqa: E402

ROLES = layout.ROLES
MS = (4, 8, 16, 32)
IN_DIMS = [layout.OBS_DIM[r] for r in ROLES]


def per_role(rows):
    pitch, in_dim = layout.fc_pitch(10), 10
    theta = torch.randn(pitch, device="cuda") * 0.05
    sig = torch.tensor([0.05], dtype=torch.float64, device="cuda")
    out = torch.empty((rows, pitch), device="cuda")
    fns = {"k5": lambda: ops.es_perturb(theta, in_dim, sig, 1, "agent_0", 0, 0, rows, out=out)}
    keep = []
    for m in MS:
        _, U, ke = _full_basis(m)
        M = (U[:, :pitch] * 20.0).contiguous()           # vectors of norm ~20 on the Linear entries
        G = (M.double() @ M.double().T).contiguous()
        c = engine.lmma_constants(rows, layout.fc_dim(in_dim), m)
        beta = torch.empty((rows, m), device="cuda")
        keep += [U, M, G, beta]
        fns[f"project_m{m}"] = (lambda M=M, G=G, c=c, m=m, beta=beta: ops.es_lmma_project(
            M, m, G, c["c_d"], in_dim, 1, "agent_0", 0, 0, rows, beta=beta))
        fns[f"lmma_k5_m{m}"] = (lambda M=M, beta=beta, c=c, m=m: ops.es_perturb_lmma(
            theta, in_dim, sig, M, m, beta, c["alpha"][m], 1, "agent_0", 0, 0, rows, out=out))
        fns[f"subspace_k5_k{m}"] = (lambda U=U[:, :pitch], kr=ke[0:1]: ops.es_perturb_subspace(
            theta, in_dim, sig, U, kr, 0.5, 1, "agent_0", 0, 0, rows, out=out))
        fns[f"project_m{m}"]()
    r = alternate(fns, 20 if rows <= 1024 else 5)
    for m in MS:
        r[f"lmma_total_m{m}"] = {"us": round(r[f"project_m{m}"]["us"] + r[f"lmma_k5_m{m}"]["us"], 1)}
    return {"rows": rows, **r}


def update(m=8, rows=1024):
    n = sum(layout.fc_pitch(d) for d in IN_DIMS)
    pitch = layout.fc_pitch(10)
    gen = torch.Generator().manual_seed(3)
    M = (torch.randn((m, n), generator=gen) * 0.1).cuda()
    p = torch.randn(n, generator=gen).cuda()
    theta = torch.randn(n, generator=gen).cuda() * 0.05
    zbar = torch.randn(n, generator=gen).cuda() * 0.05
    betabar = (torch.randn((3, m), generator=gen) * 1e-3).cuda()
    G = torch.zeros((3, m, m), dtype=torch.float64, device="cuda")
    gstate = ops.generation_state([0.05] * 3, 16, "cuda")
    cs = [engine.lmma_constants(rows, len(layout.fc_perturbable_index(d)), m) for d in IN_DIMS]
    c0 = cs[0]
    ids = torch.randperm(rows, generator=gen)[:c0["mu"]].cuda()
    w = torch.tensor(c0["w"], dtype=torch.float32).cuda()
    beta = torch.randn((rows, m), generator=gen).cuda() * 1e-3
    zb, bb = torch.empty(pitch, device="cuda"), torch.empty(m, device="cuda")
    fns = {"reduce_role": lambda: ops.es_lmma_reduce(ids, w, beta, 10, 1, "agent_0", 0, 0, rows, zbar=zb, betabar=bb),
           "apply_3_roles": lambda: ops.es_lmma_apply(
               theta, M, p, zbar, betabar, IN_DIMS, k=m, alpha=[c["alpha"][m] for c in cs],
               c_sigma=[c["c_sigma"] for c in cs], mu_w=[c["mu_w"] for c in cs], c_m=1e-6,
               c_c=[[0.0] * m for _ in cs], G=G, gstate=gstate, sigma_min=0.001, sigma_max=0.5)}
    return {"m": m, "rows": rows, "mu": c0["mu"], **alternate(fns, 20)}


def generation():
    import bench
    from coevonet_b200.MPE.fcnetwork import FCNetwork
    torch.manual_seed(0)
    theta = {r: FCNetwork(layout.OBS_DIM[r], 5, "float32").flat_row() for r in ROLES}
    engs = {}
    for name, opts in (("defaults", {}), ("lmma_m8", dict(es_distribution="lmma", es_lmma_memory=8,
                                                          learning_rate=1.0))):
        args = bench._args_bag(bench.P_PER_GPU)
        for k, v in opts.items():
            setattr(args, k, v)
        engs[name] = engine.ESEngine(args, torch.device("cuda", torch.cuda.current_device()), theta)
        for _ in range(10):                              # k = min(g, 8) = 8 from here on
            engs[name].step(sync=False)
    torch.cuda.synchronize()
    res = alternate({k: (lambda e=e: e.step(sync=False)) for k, e in engs.items()}, 10)
    for e in engs.values():
        e.check_status()
    out = {"population": bench.P_PER_GPU, "envs_per_member": bench.ENVS, "roles": 3,
           "lmma_k_eff": engs["lmma_m8"]._lmma_k()}
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
              f"forms alternated; generations: 10 per window after 10 warm-up generations (k = 8 in use)")
    res = {"card": card(), "method": method, "per_role": [per_role(1024), per_role(8192)], "update": update(),
           "generation": generation()}
    res["card_after"] = card()
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r10_es_lmma.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
