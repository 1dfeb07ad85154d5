"""Cross-generation matrix of a Co-ES run with a Hall of Fame (CIAO: current individual vs ancestral opponents).

Loads an ``engine_state_rank0.pt`` written by a run with ``--es_hof_size H --save`` and writes fp64
[filled, filled, 2] to OUT (.npy): entry [i, j] holds the mean true good-team and adversary rewards when the good team
of archive entry i plays the adversary of entry j, entries oldest first.  The generation of each entry is printed and
written to OUT with the suffix ``.generations.npy``.  A run that keeps improving shows good-team rewards that grow
along i for a fixed adversary j; cycling shows up as rows that rise and fall again.

    python scripts/hof_matrix.py ES_models/<run>/engine_state_rank0.pt --out ciao.npy [--envs 16]
"""
import argparse
import os
import sys
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from coevonet_b200 import engine, layout  # noqa: E402

ROLES = layout.ROLES


def engine_from_state(sd, device, max_evaluation_steps=None, envs=None):
    """A one-generation shell of the ES engine that holds the checkpoint's base agents and archive."""
    hof = sd.get("es_hof", engine.ES_HOF_DEFAULTS)
    if not hof["es_hof_size"]:
        raise SystemExit("the checkpoint was written without a Hall of Fame (--es_hof_size 0)")
    # the mutation powers play no part in the matrix
    args = types.SimpleNamespace(
        algorithm="ES", population=int(sd["P"]), seed=int(sd["seed"]),
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        max_evaluation_steps=max_evaluation_steps, max_timesteps_per_episode=max_evaluation_steps,
        envs_per_member=int(envs or 1), init_states="device", record_history=False, **hof,
        **sd.get("es_options", engine.ES_OPTION_DEFAULTS), **sd.get("es_distribution", engine.ES_DISTRIBUTION_DEFAULTS))
    eng = engine.ESEngine(args, device, sd["theta"])
    # only the archive matters here; the world size and shard of the run that wrote it do not
    eng.hof_ring.copy_(sd["hof_ring"])
    eng.hof_head, eng.hof_filled = int(sd["hof_head"]), int(sd["hof_filled"])
    eng.hof_slot_gen = [int(g) for g in sd["hof_slot_gen"]]
    return eng


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("checkpoint")
    ap.add_argument("--out", required=True, help="the .npy file to write")
    ap.add_argument("--envs", type=int, default=16, help="games per (good team, adversary) pair")
    ap.add_argument("--max_evaluation_steps", type=int, default=None, help="agent-step limit of a game (default 75)")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("hof_matrix.py needs a CUDA device")
    sd = torch.load(a.checkpoint, map_location="cpu", weights_only=False)
    eng = engine_from_state(sd, torch.device("cuda", 0), a.max_evaluation_steps, a.envs)
    m = eng.hof_matrix(a.envs).cpu().numpy()
    gens = np.asarray(eng.hof_generations(), dtype=np.int64)
    np.save(a.out, m)
    np.save(os.path.splitext(a.out)[0] + ".generations.npy", gens)
    print(f"{m.shape[0]} archive entries, generations {gens.tolist()}")
    print("good-team reward (rows: good team of entry i, columns: adversary of entry j):")
    print(np.array2string(m[..., 0], precision=2, max_line_width=200))
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
