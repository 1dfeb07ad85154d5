"""The Co-ES Hall of Fame on the GPU: the opponent-slot kernel against the oracle, a one-slot archive against the
default engine, K = 4 opponent sets against four separate rollouts, determinism, resume, the cross-generation matrix
against the indexed rollout, and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_hof

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 31337
GAP = 1e-4          # decision margin below which a fork is tolerated (tests/test_gpu_rollout.py)


@pytest.mark.parametrize("seed,gen,K,filled,newest", [(1870300, 0, 1, 1, 0), (1870300, 0, 5, 1, 0),
                                                      (99, 7, 6, 6, 2), (2 ** 40 + 17, 123, 9, 20, 19),
                                                      (7, 2 ** 32 - 1, 300, 1000, 500), (5, 9, 4, 2 ** 32, 7)])
def test_opponent_slots_kernel_matches_the_oracle(seed, gen, K, filled, newest):
    from coevonet_b200 import ops
    got = ops.es_hof_opponents(seed, gen, K, filled, newest, "cuda").cpu().numpy()
    assert np.array_equal(got, es_hof.opponent_slots(seed, gen, K, filled, newest))


def test_opponent_slots_kernel_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    for K, filled, newest in ((0, 4, 0), (2, 0, 0), (2, 4, 4), (2, 2 ** 32 + 1, 0)):
        with pytest.raises(_lib.CevError):
            ops.es_hof_opponents(1, 0, K, filled, newest, "cuda")


# ---------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------
def _args(P, E=4, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=8, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=E, reference_compat=True, init_states="device", seed=SEED, plots=False,
        record_history=False)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _engine(P, kernels=None, **opts):
    from coevonet_b200 import engine, layout, ops
    theta = {r: ops.fc_init(layout.OBS_DIM[r], 5, r, 0, 1, "cuda")[0].cpu() for r in ROLES}
    return engine.ESEngine(_args(P, **opts), torch.device("cuda", 0), theta, kernels=kernels)


def _bits(eng):
    eng.check_status()
    out = {"theta": eng.theta_cat.cpu().numpy().view(np.uint32), "gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["rew_" + r] = eng.rewards[r].cpu().numpy()
    if eng.hof_ring is not None:
        out["ring"] = eng.hof_ring.cpu().numpy().view(np.uint32)
    return out


def _same(a, b, keys=None):
    for k in keys or a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("init_states", ["device", "reference"], ids=["device_states", "host_states"])
def test_one_slot_archive_equals_the_default_engine(init_states):
    """H = K = 1: the same theta, rewards, fitness and evaluation games (the generation state) as the default."""
    plain = _engine(64, init_states=init_states)
    hof = _engine(64, init_states=init_states, es_hof_size=1, es_hof_opponents=1)
    for _ in range(3):
        plain.step(sync=False)
        hof.step(sync=False)
        _same(_bits(plain), _bits(hof), keys=["theta", "gstate"] + [p + r for p in ("fit_", "rew_") for r in ROLES])
    assert np.array_equal(_bits(hof)["ring"][0], _bits(hof)["theta"])
    assert plain.variant == hof.variant


class _Recording:
    """coevonet_b200.ops, recording the roles' rollout pass of the engine."""

    def __init__(self):
        from coevonet_b200 import ops
        self.ops, self.calls = ops, []

    def __getattr__(self, name):
        return getattr(self.ops, name)

    def mpe_rollout_roles(self, specs, **kw):
        outs = self.ops.mpe_rollout_roles(specs, **kw)
        self.calls.append((specs, outs, kw))
        return outs


def test_four_opponent_sets_equal_four_separate_rollouts():
    from coevonet_b200 import ops
    P, E, K = 64, 4, 4
    rec = _Recording()
    eng = _engine(P, kernels=rec, E=E, es_hof_size=6, es_hof_opponents=K)
    for _ in range(5):
        eng.step(sync=False)
    rec.calls.clear()
    eng.evaluate()
    eng.check_status()
    slots = eng.hof_ids.cpu().numpy()
    assert np.array_equal(slots, es_hof.opponent_slots(SEED, eng.gen, K, 6, (eng.hof_head - 1) % 6))
    assert len(set(slots.tolist())) > 1
    (specs, outs, kw), = rec.calls
    limit = eng.args.max_timesteps_per_episode
    n_safe = n_all = 0
    for (role, members, opp_a, opp_b, init), out in zip(specs, outs):
        assert tuple(out.shape) == (P, K, E, 4) and tuple(init.shape) == (P, K, E, 11)
        o, p = eng.cols[{"agent_0": "adversary_0", "agent_1": "adversary_0", "adversary_0": "agent_0"}[role]]
        for k in range(K):
            assert torch.equal(opp_a[k], eng.hof_ring[slots[k], o:o + p])
        per_set = [ops.mpe_rollout(role, members, opp_a[k:k + 1].contiguous(), opp_b[k:k + 1].contiguous(),
                                   init[:, k:k + 1].contiguous(), n_cycles=kw["n_cycles"], status=eng.status)
                   for k in range(K)]
        sep = torch.cat(per_set, dim=1).cpu().numpy()                       # [P, K, E, 4]
        got = out.cpu().numpy()
        safe = sep[..., 3] > GAP
        n_safe, n_all = n_safe + int(safe.sum()), n_all + safe.size
        np.testing.assert_allclose(got[..., :3][safe], sep[..., :3][safe], rtol=1e-9, atol=1e-9, err_msg=role)
        # the reward is the mean over the K x E games; members whose games are all safe match the separate calls
        assert torch.equal(eng.rewards[role], eng._role_slot(out, role, limit).mean(dim=(1, 2)))
        want = torch.stack([eng._role_slot(s, role, limit).mean(dim=(1, 2)) for s in per_set]).mean(dim=0)
        ok = torch.from_numpy(safe.reshape(P, -1).all(axis=1)).cuda()
        assert int(ok.sum()) >= P // 4, role
        torch.testing.assert_close(eng.rewards[role][ok], want[ok], rtol=1e-9, atol=1e-9)
    assert n_safe >= 0.8 * n_all
    eng.check_status()


def test_hof_engine_deterministic_and_resume_bit_exact(tmp_path):
    kw = dict(es_hof_size=3, es_hof_opponents=2, mirrored_sampling=True, fitness_shaping="centered_rank")
    runs = []
    for _ in range(2):
        eng = _engine(64, **kw)
        for _ in range(5):
            eng.step(sync=False)
        runs.append(_bits(eng))
    _same(*runs)
    first = _engine(64, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "hof.pt")
    second = _engine(64, **kw)
    second.load_state_dict(torch.load(tmp_path / "hof.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    _same(runs[0], _bits(second))


def test_hof_matrix_equals_the_indexed_rollout_per_pair():
    from coevonet_b200 import ops
    eng = _engine(32, es_hof_size=4, es_hof_opponents=2)
    for _ in range(5):                                    # wrapped: slot order differs from generation order
        eng.step(sync=False)
    E = 8
    m = eng.hof_matrix(E).cpu().numpy()
    n = eng.hof_filled
    assert m.shape == (n, n, 2) and m.dtype == np.float64
    gens = eng.hof_generations()
    slot_of = {g: s for s, g in enumerate(eng.hof_slot_gen)}
    rows = eng.hof_ring[[slot_of[g] for g in gens]]                       # oldest first
    w = {r: rows[:, o:o + p].contiguous() for r, (o, p) in eng.cols.items()}
    # episode (j, i, e): the adversary of entry j against the good team of entry i, the matrix's init records
    jj, ii, _ = np.meshgrid(np.arange(n), np.arange(n), np.arange(E), indexing="ij")
    idx = torch.from_numpy(np.stack([jj.ravel(), ii.ravel(), ii.ravel()], axis=1).astype(np.int32)).cuda()
    init = ops.init_states(SEED, eng._hof_matrix_tag, n * n * E, "cuda")
    out = ops.mpe_rollout_indexed(w["adversary_0"], w["agent_0"], w["agent_1"], idx, init,
                                  n_cycles=ops.cycles_for_limit(400), status=eng.status)
    eng.check_status()
    out = out.cpu().numpy().reshape(n, n, E, 4)
    safe = (out[..., 3] > GAP).all(axis=2)                                # [j, i]
    assert safe.sum() >= 0.5 * safe.size
    for j in range(n):
        for i in range(n):
            if safe[j, i]:
                np.testing.assert_allclose(m[i, j], out[j, i][:, [0, 2]].mean(axis=0), rtol=1e-9, atol=1e-9)


# ---------------------------------------------------------------------------------------------------------------
# two GPUs
# ---------------------------------------------------------------------------------------------------------------
def _worker(rank, world, P, E, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from coevonet_b200 import engine, layout, ops
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    comm = engine.Comm()
    theta = {r: ops.fc_init(layout.OBS_DIM[r], 5, r, 0, 1, dev)[0].cpu() for r in ROLES}
    eng = engine.ESEngine(_args(P, E, es_hof_size=2, es_hof_opponents=2), dev, theta, comm=comm)
    for _ in range(2):
        eng.step(sync=False)
    eng.evaluate()
    out = dict(rewards=np.stack([comm.all_gather_rows(eng.rewards[r], eng.shard).cpu().numpy() for r in ROLES]),
               ring=eng.hof_ring.cpu().numpy(), ids=eng.hof_ids.cpu().numpy())
    q.put((rank, out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _launch(world, P, E, port):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, P, E, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return [outs[r] for r in range(world)]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_hof_sharded_over_two_gpus_equal_one_gpu():
    P, E = 387, 16                                 # 194 + 193 rows
    one = _launch(1, P, E, 29731)[0]
    two = _launch(2, P, E, 29732)
    assert np.array_equal(two[0]["ring"], two[1]["ring"])              # replicas agree
    for o in two:
        assert np.array_equal(o["ids"], one["ids"])
        # the all-reduce adds the ranks' partial updates in another order: fp32 rounding in theta only
        np.testing.assert_allclose(o["ring"], one["ring"], rtol=0, atol=1e-5)
