"""The Co-ES Hall of Fame on the host: the opponent-slot draw of the oracle against a scalar restatement, flag
validation, and the ES engine's Hall-of-Fame path with the checker backend (tests/es_hof_backend.py): the archive
ring, the opponents handed to the rollout, H = K = 1 against the default engine, resume, checkpoints, the
cross-generation matrix and two gloo ranks."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_hof, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
HOF = dict(es_hof_size=3, es_hof_opponents=2)


# ---------------------------------------------------------------------------------------------------------------
# the draw
# ---------------------------------------------------------------------------------------------------------------
def _scalar_slots(seed, gen, K, filled, newest):
    """One Philox call per set, straight from the header's formula."""
    k0, k1 = philox.split_seed(seed)
    out = [newest]
    for k in range(1, K):
        block = philox.philox4x32_10(np.uint32((k - 1) >> 2), np.uint32(0), np.uint32(gen),
                                     np.uint32(es_hof.KIND_HOF << 8), k0, k1)
        w = int(block[(k - 1) & 3])
        out.append((w * filled) >> 32)
    return out


@pytest.mark.parametrize("seed,gen,filled,K", [(1870300, 0, 1, 1), (1870300, 0, 1, 7), (99, 5, 6, 6),
                                               (2 ** 40 + 17, 123, 20, 9), (7, 2 ** 32 - 1, 1000, 33),
                                               (5, 9, 2 ** 32, 4)])
def test_oracle_draw_is_the_documented_formula(seed, gen, filled, K):
    newest = (gen % filled)
    got = es_hof.opponent_slots(seed, gen, K, filled, newest)
    assert got.dtype == np.int64 and got.shape == (K,)
    assert got.tolist() == _scalar_slots(seed, gen, K, filled, newest)
    assert got[0] == newest and np.all((got >= 0) & (got < filled))


def test_draw_is_uniform_and_keyed_by_seed_and_generation():
    from scipy import stats
    filled, K = 10, 4001
    slots = es_hof.opponent_slots(3, 4, K, filled, 9)[1:]
    counts = np.bincount(slots, minlength=filled)
    assert stats.chisquare(counts).pvalue > 1e-3
    assert not np.array_equal(slots, es_hof.opponent_slots(3, 5, K, filled, 9)[1:])
    assert not np.array_equal(slots, es_hof.opponent_slots(4, 4, K, filled, 9)[1:])
    # a longer draw starts with the shorter one
    assert np.array_equal(es_hof.opponent_slots(3, 4, 10, filled, 9), es_hof.opponent_slots(3, 4, K, filled, 9)[:10])


def test_oracle_ring_bookkeeping():
    ring = es_hof.Ring(3, np.full(4, 0.0))
    assert (ring.head, ring.filled, ring.newest) == (1, 1, 0)
    for g in range(1, 6):
        ring.append(np.full(4, float(g)), g)
        assert ring.filled == min(g + 1, 3) and ring.head == (g + 1) % 3
        assert ring.rows[ring.newest][0] == g and ring.slot_gen[ring.newest] == g
    assert sorted(ring.slot_gen.tolist()) == [3, 4, 5]


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_hof_flags_defaults_and_parsing():
    from coevonet_b200.engine import ES_HOF_DEFAULTS, es_hof as validate
    a = _cli(["--algorithm=ES"])
    assert (a.es_hof_size, a.es_hof_opponents) == (0, 1)
    assert validate(a) == ES_HOF_DEFAULTS
    assert validate(types.SimpleNamespace(population=4)) == ES_HOF_DEFAULTS             # attributes absent
    a = _cli(["--algorithm=ES", "--es_hof_size=8", "--es_hof_opponents=4"])
    assert validate(a) == {"es_hof_size": 8, "es_hof_opponents": 4}
    assert validate(_cli(["--algorithm=ES", "--es_hof_size=1"])) == {"es_hof_size": 1, "es_hof_opponents": 1}


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=GA", "--es_hof_size=4"], "GA"),
    (["--algorithm=GA", "--es_hof_size=4", "--es_hof_opponents=2"], "GA"),
    (["--algorithm=GA", "--es_hof_opponents=2"], "GA"),
    (["--algorithm=ES", "--es_hof_size=4", "--es_hof_opponents=5"], r"\[1, es_hof_size"),
    (["--algorithm=ES", "--es_hof_size=4", "--es_hof_opponents=0"], r"\[1, es_hof_size"),
    (["--algorithm=ES", "--es_hof_size=4", "--es_hof_opponents=-1"], r"\[1, es_hof_size"),
    (["--algorithm=ES", "--es_hof_size=-1"], ">= 0"),
    (["--algorithm=ES", "--es_hof_opponents=2"], "needs an archive"),
])
def test_hof_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_ga_engine_refuses_the_hall_of_fame_options():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="GA"):
        engine.GAEngine(_args(4, algorithm="GA", es_hof_size=2), "cpu", {}, {}, {}, kernels=_backend())


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import es_hof_backend
    return es_hof_backend


class _Recording:
    """The checker backend, recording the rollouts the engine asks for."""

    def __init__(self):
        self.rollouts = []

    def __getattr__(self, name):
        return getattr(_backend(), name)

    def mpe_rollout(self, role, members, opp_a, opp_b, init, **kw):
        self.rollouts.append((role, opp_a.clone(), opp_b.clone(), tuple(init.shape)))
        return _backend().mpe_rollout(role, members, opp_a, opp_b, init, **kw)


def _args(P, record_history=True, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=8, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.04, mutation_power_adversary=0.03,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=1, reference_compat=True, init_states="device", seed=99, plots=False,
        record_history=record_history)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _theta(seed=700):
    from coevonet_b200 import layout
    from oracle import weights
    theta = {}
    for i, r in enumerate(ROLES):
        in_dim = layout.OBS_DIM[r]
        row = np.zeros(layout.fc_pitch(in_dim), dtype=np.float32)
        row[:layout.fc_dim(in_dim)] = weights.make_fc_rows(1, in_dim, seed + i, ln_jitter=0.02)[0]
        theta[r] = torch.from_numpy(row)
    return theta


def _engine(P, comm=None, kernels=None, **kw):
    from coevonet_b200 import engine
    return engine.ESEngine(_args(P, **kw), "cpu", _theta(), kernels=kernels or _backend(), comm=comm)


def test_default_engine_has_no_archive():
    eng = _engine(4)
    assert eng.K == 1 and eng.hof_ring is None
    eng.step()
    assert eng.history[0]["hof_ids"] is None
    sd = eng.state_dict()
    assert sd["es_hof"] == {"es_hof_size": 0, "es_hof_opponents": 1} and "hof_ring" not in sd


def test_ring_and_opponents_follow_the_oracle():
    """H = 3, K = 2 over H + 2 = 5 generations: the ring, head and filled after every generation, and the opponent
    rows of every rollout, against the oracle's ring and draw."""
    H, K = 3, 2
    rec = _Recording()
    eng = _engine(4, kernels=rec, es_hof_size=H, es_hof_opponents=K)
    ring = es_hof.Ring(H, eng.theta_cat.numpy().copy())
    assert np.array_equal(eng.hof_ring.numpy(), ring.rows)
    for g in range(H + 2):
        slots = es_hof.opponent_slots(99, g, K, ring.filled, ring.newest)
        want = ring.rows[slots]
        rec.rollouts.clear()
        eng.step()
        evals = [x for x in rec.rollouts if x[3] == (1, 1, 10, 11)]          # the evaluation games: base rows only
        assert len(evals) == 1 and len(rec.rollouts) == 4
        for role, opp_a, opp_b, init_shape in rec.rollouts:
            if init_shape == (1, 1, 10, 11):
                continue
            assert init_shape == (4, K, 1, 11)
            seats = {"agent_0": ("adversary_0", "agent_1"), "agent_1": ("adversary_0", "agent_0"),
                     "adversary_0": ("agent_0", "agent_1")}[role]
            for got, r in zip((opp_a, opp_b), seats):
                o, p = eng.cols[r]
                assert np.array_equal(got.numpy(), want[:, o:o + p]), (g, role, r)
        h_slots, h_gens = eng.history[g]["hof_ids"]
        assert h_slots.tolist() == slots.tolist()
        assert h_gens.tolist() == ring.slot_gen[slots].tolist()
        ring.append(eng.theta_cat.numpy().copy(), g + 1)
        assert (eng.hof_head, eng.hof_filled) == (ring.head, ring.filled) and eng.hof_filled == min(g + 2, H)
        assert np.array_equal(eng.hof_ring.numpy(), ring.rows)
        assert eng.hof_slot_gen == ring.slot_gen.tolist()
        # set 0 is always the base agents the generation started from
        assert ring.slot_gen[slots[0]] == g


@pytest.mark.parametrize("init_states", ["device", "reference"], ids=["device_states", "host_states"])
def test_one_slot_archive_equals_the_default_engine(init_states):
    a = _engine(4, init_states=init_states)
    b = _engine(4, init_states=init_states, es_hof_size=1, es_hof_opponents=1)
    for g in range(3):
        ea, eb = a.step(), b.step()
        assert ea == eb
        for r in ROLES:
            assert np.array_equal(a.history[g]["rewards"][r], b.history[g]["rewards"][r])
            assert np.array_equal(a.history[g]["delta"][r], b.history[g]["delta"][r])
        assert torch.equal(a.theta_cat, b.theta_cat) and torch.equal(b.hof_ring[0], b.theta_cat)
    assert torch.equal(a.gstate, b.gstate)


def test_reward_is_the_mean_over_the_opponent_sets():
    """With K = 2 each member's reward is the mean of its games against the two sets."""
    rec = _Recording()
    eng = _engine(4, kernels=rec, es_hof_size=2, es_hof_opponents=2, record_history=False)
    eng.step(sync=False)                                  # generation 1 draws from two distinct snapshots
    rec.rollouts.clear()
    be = _backend()
    eng.evaluate()
    limit = eng.args.max_timesteps_per_episode
    assert len(rec.rollouts) == 3
    for role, opp_a, opp_b, _ in rec.rollouts:
        init = eng._initial_states(eng.P, 2, eng.shard, ROLES.index(role) + 4 * eng.gen)
        per_set = []
        for k in range(2):
            out = be.mpe_rollout(role, eng.members[role], opp_a[k:k + 1], opp_b[k:k + 1], init[:, k:k + 1],
                                 n_cycles=be.cycles_for_limit(limit))
            per_set.append(eng._role_slot(out, role, limit).mean(dim=(1, 2)))
        assert torch.allclose(eng.rewards[role], (per_set[0] + per_set[1]) / 2, rtol=1e-12, atol=1e-12)


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(HOF, record_history=False)
    full = _engine(4, **kw)
    for _ in range(5):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "hof.pt")
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(tmp_path / "hof.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.theta_cat, full.theta_cat)
    assert torch.equal(second.hof_ring, full.hof_ring)
    assert (second.hof_head, second.hof_filled, second.hof_slot_gen) == \
        (full.hof_head, full.hof_filled, full.hof_slot_gen)


def test_resume_refuses_other_hof_settings():
    hof = _engine(4, record_history=False, **HOF)
    hof.step(sync=False)
    sd = hof.state_dict()
    with pytest.raises(ValueError, match="Hall of Fame"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="Hall of Fame"):
        _engine(4, record_history=False, es_hof_size=3, es_hof_opponents=3).load_state_dict(sd)
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    with pytest.raises(ValueError, match="Hall of Fame"):
        _engine(4, record_history=False, **HOF).load_state_dict(plain.state_dict())
    # a checkpoint without the settings (written before they existed) has no Hall of Fame
    old = plain.state_dict()
    del old["es_hof"]
    fresh = _engine(4, record_history=False)
    fresh.load_state_dict(old)
    assert torch.equal(fresh.theta_cat, plain.theta_cat)
    with pytest.raises(ValueError, match="Hall of Fame"):
        _engine(4, record_history=False, **HOF).load_state_dict(old)


def test_hof_matrix_equals_per_pair_rollouts():
    eng = _engine(4, record_history=False, es_hof_size=3, es_hof_opponents=2)
    for _ in range(4):                                    # the ring has wrapped: slot order != generation order
        eng.step(sync=False)
    gens = eng.hof_generations()
    assert gens == [2, 3, 4]
    E = 2
    m = eng.hof_matrix(E)
    assert m.dtype == torch.float64 and tuple(m.shape) == (3, 3, 2)
    be = _backend()
    slot_of = {g: s for s, g in enumerate(eng.hof_slot_gen)}
    ring = eng.hof_ring
    init = be.init_states(99, eng._hof_matrix_tag, 9 * E, "cpu").reshape(3, 3, E, 11)
    col = {r: (lambda s, o=o, p=p: ring[s:s + 1, o:o + p]) for r, (o, p) in eng.cols.items()}
    for i, gi in enumerate(gens):                         # good team of entry i
        for j, gj in enumerate(gens):                     # adversary of entry j
            si, sj = slot_of[gi], slot_of[gj]
            out = be.mpe_rollout("adversary_0", col["adversary_0"](sj), col["agent_0"](si), col["agent_1"](si),
                                 init[j:j + 1, i:i + 1], n_cycles=be.cycles_for_limit(400))
            want = out[0, 0, :, [0, 2]].mean(dim=0)
            assert torch.equal(m[i, j], want), (i, j)
    with pytest.raises(ValueError, match="es_hof_size"):
        _engine(4, record_history=False).hof_matrix()


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, es_hof_size=2, es_hof_opponents=2)
    evs = [eng.step() for _ in range(3)]
    theta_hist = [eng.hof_ring[s].numpy().copy() for s in range(2)]
    q.put(dict(rank=rank, evs=np.asarray(evs),
               rewards=np.stack([eng.history[g]["rewards"][r] for g in range(3) for r in ROLES]),
               slots=np.stack([eng.history[g]["hof_ids"][0] for g in range(3)]),
               theta=eng.theta_cat.numpy().copy(), ring=np.stack(theta_hist),
               newest_is_theta=bool(np.array_equal(theta_hist[(eng.hof_head - 1) % 2], eng.theta_cat.numpy()))))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _launch(world, P, port):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_run, args=(r, world, P, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = [q.get(timeout=600) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    return sorted(outs, key=lambda o: o["rank"])


@pytest.mark.timeout(900)
def test_hof_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows; the archive and the draws are replicated."""
    P = 5
    single = _launch(1, P, 29651)[0]
    two = _launch(2, P, 29652)
    for o in two:
        assert np.array_equal(o["slots"], single["slots"])
        assert o["newest_is_theta"]
        # generation 0 plays identical founders and snapshots
        assert np.array_equal(o["rewards"][:3], single["rewards"][:3])
        np.testing.assert_allclose(o["rewards"], single["rewards"], rtol=1e-12, atol=0)
        # the two ranks' partial updates are added in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["ring"], single["ring"], rtol=0, atol=3e-5)
    for k in ("theta", "ring", "rewards"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree bit for bit
