"""Co-ES novelty search on the host: the oracle's probe observations against the environment, its k-NN novelty against
a brute-force restatement, flag validation, and the ES engine's novelty path with the checker backend
(tests/es_novelty_backend.py): the default call log at w = 0, the archive rings over A + 2 generations, the combined
fitness, resume, checkpoints and two gloo ranks."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_novelty as en, es_options as oes, mpe_env

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
NOV = dict(es_novelty_weight=0.5, es_novelty_k=2, es_novelty_archive=3, fitness_shaping="centered_rank")


# ---------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------
def test_probe_observations_are_the_environment_observations():
    states = en.probe_states(1870300)
    assert states.shape == (32, 11)
    env = mpe_env.SimpleAdversaryEnv()
    for role in ROLES:
        obs = en.probe_obs(states, role)
        assert obs.dtype == np.float32 and obs.shape == (32, 10 if role != "adversary_0" else 8)
        for i, rec in enumerate(states):
            env.load_flat_state(rec)
            assert np.array_equal(obs[i], env.observe(role)), (role, i)
    # a stream of its own: not the training states of generation 0
    from oracle import philox
    assert not np.array_equal(states, philox.init_states(1870300, 0, 32))


def _brute_novelty(x, archive, k):
    """sorted() over (distance, slot) pairs, each distance summed one term at a time in Python floats."""
    pairs = []
    for e, y in enumerate(archive):
        s = 0.0
        for t in range(len(x)):
            d = float(np.float64(x[t]) - np.float64(y[t]))
            s = s + d * d
        pairs.append((float(np.sqrt(s)), e))
    ke = min(k, len(archive))
    acc = 0.0
    for d, _ in sorted(pairs)[:ke]:
        acc += d
    return acc / ke


@pytest.mark.parametrize("filled,k", [(1, 1), (1, 10), (7, 3), (7, 7), (5, 32), (40, 10)])
def test_knn_novelty_equals_brute_force(filled, k):
    rng = np.random.default_rng(filled * 100 + k)
    bcs = rng.dirichlet(np.ones(5), size=(6, 32)).reshape(6, 160).astype(np.float32)
    archive = rng.dirichlet(np.ones(5), size=(filled, 32)).reshape(filled, 160).astype(np.float32)
    got = en.novelty(bcs, archive, k)
    assert got.dtype == np.float64
    for i in range(6):
        assert got[i] == _brute_novelty(bcs[i], archive, k), i


def test_knn_novelty_with_ties():
    rng = np.random.default_rng(3)
    base = rng.random((4, 160)).astype(np.float32)
    archive = np.concatenate([base, base, base[:2]])             # every distance appears two or three times
    bcs = np.concatenate([base[:2], rng.random((2, 160)).astype(np.float32)])
    for k in (1, 2, 3, 5, 10):
        got = en.novelty(bcs, archive, k)
        for i in range(4):
            assert got[i] == _brute_novelty(bcs[i], archive, k)
    # a member equal to three entries: its three nearest distances are 0
    assert en.novelty(base[:1], archive, 3)[0] == 0.0


def test_combination_formula():
    rng = np.random.default_rng(5)
    R, N = rng.standard_normal(9), rng.standard_normal(9)
    cr, cn = oes.centered_ranks(R), oes.centered_ranks(N)
    assert np.array_equal(en.combine(cr, cn, 1.0), cn)
    assert np.array_equal(en.combine(cr, cn, 0.5), 0.5 * cr + 0.5 * cn)
    w = 0.3
    assert np.array_equal(en.combine(cr, cn, w), (1.0 - w) * cr + w * cn)


def test_oracle_ring_bookkeeping():
    ring = en.Ring(3, np.full(160, 0.0, np.float32))
    assert (ring.head, ring.filled) == (1, 1)
    for g in range(1, 6):
        ring.append(np.full(160, float(g), np.float32))
        assert ring.filled == min(g + 1, 3) and ring.head == (g + 1) % 3
    assert sorted(ring.rows[:, 0].tolist()) == [3.0, 4.0, 5.0]


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_novelty_flags_defaults_and_parsing():
    from coevonet_b200.engine import ES_NOVELTY_DEFAULTS, es_novelty as validate
    a = _cli(["--algorithm=ES"])
    assert (a.es_novelty_weight, a.es_novelty_k, a.es_novelty_archive) == (0.0, None, None)
    assert validate(a) == ES_NOVELTY_DEFAULTS
    assert validate(types.SimpleNamespace(population=4)) == ES_NOVELTY_DEFAULTS            # attributes absent
    assert validate(_cli(["--algorithm=ES", "--es_novelty_weight=1", "--fitness_shaping=centered_rank"])) == \
        {"es_novelty_weight": 1.0, "es_novelty_k": 10, "es_novelty_archive": 1024}
    assert validate(_cli(["--algorithm=ES", "--es_novelty_weight=0.5", "--es_novelty_k=32", "--es_novelty_archive=1",
                          "--fitness_shaping=centered_rank"])) == \
        {"es_novelty_weight": 0.5, "es_novelty_k": 32, "es_novelty_archive": 1}
    # with the other Co-ES options
    assert validate(_cli(["--algorithm=ES", "--es_novelty_weight=0.5", "--fitness_shaping=centered_rank",
                          "--mirrored_sampling", "--es_hof_size=2", "--es_subspace_dim=2", "--es_optimizer=adam",
                          "--es_novelty_archive=32768"]))["es_novelty_archive"] == 32768
    assert validate(_cli(["--algorithm=GA", "--es_novelty_weight=0"])) == ES_NOVELTY_DEFAULTS


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=GA", "--es_novelty_weight=0.5", "--fitness_shaping=centered_rank"], "GA"),
    (["--algorithm=GA", "--es_novelty_k=4"], "GA"),
    (["--algorithm=GA", "--es_novelty_archive=4"], "GA"),
    (["--algorithm=ES", "--es_novelty_weight=1.5", "--fitness_shaping=centered_rank"], r"\[0, 1\]"),
    (["--algorithm=ES", "--es_novelty_weight=-0.1", "--fitness_shaping=centered_rank"], r"\[0, 1\]"),
    (["--algorithm=ES", "--es_novelty_weight=nan", "--fitness_shaping=centered_rank"], r"\[0, 1\]"),
    (["--algorithm=ES", "--es_novelty_k=4"], "needs es_novelty_weight"),
    (["--algorithm=ES", "--es_novelty_archive=64"], "needs es_novelty_weight"),
    (["--algorithm=ES", "--es_novelty_weight=0", "--es_novelty_k=10"], "needs es_novelty_weight"),
    (["--algorithm=ES", "--es_novelty_weight=0.5", "--es_novelty_k=0", "--fitness_shaping=centered_rank"],
     r"\[1, 32\]"),
    (["--algorithm=ES", "--es_novelty_weight=0.5", "--es_novelty_k=33", "--fitness_shaping=centered_rank"],
     r"\[1, 32\]"),
    (["--algorithm=ES", "--es_novelty_weight=0.5", "--es_novelty_archive=0", "--fitness_shaping=centered_rank"],
     r"\[1, 32768\]"),
    (["--algorithm=ES", "--es_novelty_weight=0.5", "--es_novelty_archive=32769", "--fitness_shaping=centered_rank"],
     r"\[1, 32768\]"),
    (["--algorithm=ES", "--es_novelty_weight=0.5"], "centered_rank"),
    (["--algorithm=ES", "--es_novelty_weight=1", "--fitness_shaping=none"], "centered_rank"),
])
def test_novelty_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_engines_refuse_bad_novelty_settings():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="GA"):
        engine.GAEngine(_args(4, algorithm="GA", es_novelty_weight=0.5), "cpu", {}, {}, {}, kernels=_backend())
    with pytest.raises(ValueError, match="centered_rank"):
        _engine(4, es_novelty_weight=0.5)


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import es_novelty_backend
    return es_novelty_backend


class _Log:
    """The checker backend, logging the name of every call the engine makes."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(_backend(), name)
        if not callable(fn):
            return fn

        def logged(*a, **kw):
            self.calls.append(name)
            return fn(*a, **kw)
        return logged


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


def test_zero_weight_issues_the_default_calls():
    logs = []
    for kw in ({}, {"es_novelty_weight": 0.0}, {"es_novelty_weight": 0, "fitness_shaping": "none"}):
        log = _Log()
        eng = _engine(4, kernels=log, **kw)
        for _ in range(2):
            eng.step()
        assert eng.novelty_ring is None and eng.history[0]["novelty"] is None
        assert eng.history[1]["novelty_filled"] is None
        logs.append(log.calls)
    assert logs[0] == logs[1] == logs[2] and "es_perturb" in logs[0]
    assert not any("novelty" in c for c in logs[0])
    sd = eng.state_dict()
    assert sd["es_novelty"] == {"es_novelty_weight": 0.0, "es_novelty_k": None, "es_novelty_archive": None}
    assert "novelty_ring" not in sd


@pytest.mark.parametrize("w", [1.0, 0.5], ids=["ns", "nsr"])
def test_ring_novelty_and_fitness_follow_the_oracle(w):
    """A = 3 over A + 2 = 5 generations: the probe observations, every generation's novelty (members against the
    ring as it stood), the combined fitness the update used, and the rings, head and filled after every
    generation, against the oracle."""
    from coevonet_b200 import layout
    A, k = 3, 2
    eng = _engine(4, es_novelty_weight=w, es_novelty_k=k, es_novelty_archive=A, fitness_shaping="centered_rank")
    states = en.probe_states(99)
    obs = {r: en.probe_obs(states, r) for r in ROLES}
    for r in ROLES:
        assert np.array_equal(eng.novelty_probe_obs[r].numpy(), obs[r])

    def theta_bc(role):
        o, p = eng.cols[role]
        return en.bc(eng.theta_cat.numpy()[None, o:o + p], layout.OBS_DIM[role], obs[role])[0]

    rings = {r: en.Ring(A, theta_bc(r)) for r in ROLES}
    for g in range(A + 2):
        filled = rings[ROLES[0]].filled
        eng.step()
        h = eng.history[g]
        assert h["novelty_filled"] == filled
        for i, r in enumerate(ROLES):
            in_dim = layout.OBS_DIM[r]
            bcs = en.bc(eng.members[r].numpy(), in_dim, obs[r])
            want = en.novelty(bcs, rings[r].rows[:rings[r].filled], k)
            assert np.array_equal(h["novelty"][r], want), (g, r)
            reward = eng.fitness[r].numpy()
            F = en.combine(oes.centered_ranks(reward), oes.centered_ranks(want), w)
            assert np.array_equal(h["shaped_fitness"][r], F), (g, r)
            rings[r].append(theta_bc(r))
            assert np.array_equal(eng.novelty_ring[i].numpy(), rings[r].rows), (g, r)
        assert (eng.novelty_head, eng.novelty_filled) == (rings[ROLES[0]].head, rings[ROLES[0]].filled)
        assert eng.novelty_filled == min(g + 2, A)
    # the ring has wrapped: slot 0 holds the base agents after generation 2, not the founders
    assert rings[ROLES[0]].head == (A + 3) % A


def test_novelty_changes_the_update():
    """w = 1 weights the members by their novelty ranks alone: another update than the reward's ranks."""
    a = _engine(4, fitness_shaping="centered_rank")
    b = _engine(4, es_novelty_weight=1.0, fitness_shaping="centered_rank")
    a.step()
    b.step()
    for r in ROLES:
        assert np.array_equal(a.history[0]["rewards"][r], b.history[0]["rewards"][r])
        assert np.array_equal(b.history[0]["shaped_fitness"][r], oes.centered_ranks(b.history[0]["novelty"][r]))
    assert not torch.equal(a.theta_cat, b.theta_cat)


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(NOV, record_history=False)
    full = _engine(4, **kw)
    for _ in range(5):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "nov.pt")
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(tmp_path / "nov.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.theta_cat, full.theta_cat)
    assert torch.equal(second.novelty_ring, full.novelty_ring)
    assert (second.novelty_head, second.novelty_filled) == (full.novelty_head, full.novelty_filled)
    for r in ROLES:
        assert torch.equal(second.novelty[r], full.novelty[r])


def test_resume_refuses_other_novelty_settings():
    nov = _engine(4, record_history=False, **NOV)
    nov.step(sync=False)
    sd = nov.state_dict()
    assert sd["es_novelty"] == {"es_novelty_weight": 0.5, "es_novelty_k": 2, "es_novelty_archive": 3}
    assert sd["novelty_filled"] == 2 and tuple(sd["novelty_ring"].shape) == (3, 3, 160)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, fitness_shaping="centered_rank").load_state_dict(sd)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **dict(NOV, es_novelty_k=3)).load_state_dict(sd)
    plain = _engine(4, record_history=False, fitness_shaping="centered_rank")
    plain.step(sync=False)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **NOV).load_state_dict(plain.state_dict())
    # a checkpoint without the settings (written before they existed) loads as off
    old = plain.state_dict()
    del old["es_novelty"]
    fresh = _engine(4, record_history=False, fitness_shaping="centered_rank")
    fresh.load_state_dict(old)
    assert torch.equal(fresh.theta_cat, plain.theta_cat)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **NOV).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **NOV)
    theta0, ring0 = eng.theta_cat.numpy().copy(), eng.novelty_ring.numpy().copy()
    evs = [eng.step() for _ in range(3)]
    q.put(dict(rank=rank, evs=np.asarray(evs),
               novelty=np.stack([eng.history[g]["novelty"][r] for g in range(3) for r in ROLES]),
               F=np.stack([eng.history[g]["shaped_fitness"][r] for g in range(3) for r in ROLES]),
               theta0=theta0, ring0=ring0, theta=eng.theta_cat.numpy().copy(), ring=eng.novelty_ring.numpy().copy()))
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
def test_novelty_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows; the rings are replicated without a collective."""
    P = 5
    single = _launch(1, P, 29671)[0]
    two = _launch(2, P, 29672)
    for o in two:
        # generation 0: the same base agents and founders' ring, so the same members, novelty and fitness
        assert np.array_equal(o["theta0"], single["theta0"]) and np.array_equal(o["ring0"], single["ring0"])
        assert np.array_equal(o["novelty"][:3], single["novelty"][:3])
        assert np.array_equal(o["F"][:3], single["F"][:3])
        # the two ranks' partial updates are added in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["ring"], single["ring"], rtol=0, atol=1e-4)
        np.testing.assert_allclose(o["novelty"], single["novelty"], rtol=1e-3, atol=1e-5)
    for k in ("theta", "ring", "novelty", "F"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree bit for bit
