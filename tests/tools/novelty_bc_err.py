"""Largest |kernel - oracle| of the novelty search's behaviour characterisation (cev_novelty_bc_f32 against the NumPy
fp32 forward of oracle/es_novelty.py), over sigma-0.05 members of each role, at 1,024 members (development aid).
Writes <out-dir>/r07_es_novelty_bc_error.json with the card it ran on.

    python tests/tools/novelty_bc_err.py --out-dir OUT
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from coevonet_b200 import layout, ops  # noqa: E402
from oracle import es_novelty as en  # noqa: E402

P, SEED = 1024, 11


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out-dir", required=True)
    ns = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    res = {"card": q.stdout.strip() or q.stderr.strip(), "members_per_role": P, "sigma": 0.05, "error": {}}
    obs_all = ops.init_states(SEED, en.PROBE_TAG, en.PROBES, "cuda")
    for role in layout.ROLES:
        in_dim = layout.OBS_DIM[role]
        theta = ops.fc_init(in_dim, SEED, role, 0, 1, "cuda")[0]
        members = ops.es_perturb(theta, in_dim, 0.05, SEED, role, 0, 0, P)
        obs = ops.novelty_probe_obs(obs_all, role)
        got = ops.novelty_bc(members, in_dim, obs).cpu().numpy()
        want = en.bc(members.cpu().numpy()[:, :layout.fc_dim(in_dim)], in_dim, obs.cpu().numpy())
        err = np.abs(got.astype(np.float64) - want.astype(np.float64))
        res["error"][role] = {"max_abs": float(err.max()), "mean_abs": float(err.mean()),
                              "exact_fraction": float((err == 0).mean())}
    os.makedirs(ns.out_dir, exist_ok=True)
    with open(os.path.join(ns.out_dir, "r07_es_novelty_bc_error.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
