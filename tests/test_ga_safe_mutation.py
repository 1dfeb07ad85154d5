"""Co-GA safe mutations (SM-G-SUM) on the host: the oracle's fp64 backpropagation against torch.autograd, the scale
rule and the children, flag validation, and the GA engine's safe-mutation path with the checker backend
(tests/ga_safe_mutation_backend.py): the default call log, the children against the oracle over several generations,
resume, checkpoints and two gloo ranks."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_novelty as en, ga_es, ga_safe_mutation as gsm, layout as olayout, philox, weights

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SAFE = dict(ga_safe_mutation=True, ga_safe_mutation_floor=0.05)


# ---------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------
def _autograd_G(row, in_dim, obs):
    """G [5, D] with torch.autograd on a float64 nn.Sequential mirror of the FCNetwork, one backward per logit."""
    nn = torch.nn
    p = olayout.unpack_fc(row, in_dim)
    net = nn.Sequential(nn.Linear(in_dim, 512), nn.LayerNorm(512, eps=gsm.LN_EPS), nn.ReLU(),
                        nn.Linear(512, 256), nn.LayerNorm(256, eps=gsm.LN_EPS), nn.ReLU(), nn.Linear(256, 5)).double()
    names = ["fc1.weight", "fc1.bias", "ln1.weight", "ln1.bias", "fc2.weight", "fc2.bias", "ln2.weight", "ln2.bias",
             "output.weight", "output.bias"]
    params = list(net.parameters())
    with torch.no_grad():
        for t, n in zip(params, names):
            t.copy_(torch.from_numpy(p[n].astype(np.float64)))
    y = net(torch.from_numpy(np.asarray(obs, np.float32).astype(np.float64)))
    G = []
    for k in range(5):
        grads = torch.autograd.grad(y[:, k].sum(), params, retain_graph=True)
        G.append(torch.cat([g.reshape(-1) for g in grads]).numpy())
    return np.stack(G)


def _rows_scaled(in_dim, seed):
    D = olayout.fc_dim(in_dim)
    rows = weights.make_fc_rows(5, in_dim, seed, ln_jitter=0.05)
    segs = {name: (off, int(np.prod(shape))) for name, off, shape, _ in olayout.fc_segments(in_dim)[0]}
    for i, (name, f) in enumerate((("ln1.weight", 40.0), ("ln1.weight", 0.02), ("fc2.weight", 250.0),
                                   ("fc2.weight", 0.01))):
        off, n = segs[name]
        rows[i + 1, off:off + n] = (rows[i + 1, off:off + n] * np.float32(f)).astype(np.float32)
    assert rows.shape[1] == D
    return rows


@pytest.mark.parametrize("in_dim,role", [(8, "adversary_0"), (10, "agent_0")])
def test_backprop_equals_autograd(in_dim, role):
    obs = en.probe_obs(en.probe_states(11), role)
    for row in _rows_scaled(in_dim, 300 + in_dim):
        G = gsm.gradients(row, in_dim, obs)
        want = _autograd_G(row, in_dim, obs)
        assert G.shape == want.shape == (5, olayout.fc_dim(in_dim))
        for k in range(5):
            np.testing.assert_allclose(G[k], want[k], rtol=1e-12, atol=1e-12 * np.abs(want[k]).max())
        s, mag, margin = gsm.sensitivity(row, in_dim, obs)
        np.testing.assert_allclose(s, np.sqrt((want ** 2).sum(axis=0)), rtol=1e-12, atol=1e-12 * s.max())
        assert np.all(mag >= s * (1 - 1e-12)) and margin > 0


def test_scale_rule_zero_and_floor():
    s = np.array([0.0, 1e-9, 0.01, 0.02, 5.0, 3.0e7])
    c = gsm.scale_from_s(s, 0.02)
    assert c.dtype == np.float32
    assert c[0] == 1.0
    assert c[1] == c[2] == c[3] == np.float32(1) / np.float32(0.02)
    assert c[4] == np.float32(1) / np.float32(5.0) and c[5] == np.float32(1) / np.float32(3.0e7)


def test_dead_unit_keeps_the_plain_mutation():
    """A layer-2 unit off on every probe: its out.weight column and its ln2 entries have s = 0, so c = 1."""
    in_dim = 10
    row = weights.make_fc_rows(1, in_dim, 5, ln_jitter=0.02)[0]
    segs = {name: off for name, off, _, _ in olayout.fc_segments(in_dim)[0]}
    u = 17
    row[segs["ln2.weight"] + u] = 0.0
    row[segs["ln2.bias"] + u] = -1.0
    obs = en.probe_obs(en.probe_states(3), "agent_0")
    c = gsm.scale_rows(row[None], in_dim, obs, 0.01)[0]
    assert c[segs["ln2.weight"] + u] == 1.0 and c[segs["ln2.bias"] + u] == 1.0
    assert all(c[segs["output.weight"] + k * 256 + u] == 1.0 for k in range(5))
    assert c[segs["output.bias"]] == np.float32(1) / np.float32(32)


def test_children_with_ones_equal_k3():
    """A scale row of ones gives the K3 children bit for bit, with and without crossover."""
    D = olayout.fc_dim(8)
    elites = weights.make_fc_rows(3, 8, 9)
    members = np.arange(0, 40)
    z = philox.normals(5, philox.KIND_GA, 2, 4, members, D)
    ones = np.ones((3, D), np.float32)
    for rate in (0.0, 0.7):
        want = ga_es.ga_repopulate_crossover(elites, 0.05, z, rate, 5, 2, 4, members)
        got = gsm.children(elites, ones, 0.05, z, members, rate, 5, 2, 4)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), rate


def test_children_take_the_scale_of_their_elite():
    D = olayout.fc_dim(8)
    elites = weights.make_fc_rows(2, 8, 9)
    scale = np.stack([np.full(D, 0.5, np.float32), np.full(D, 4.0, np.float32)])
    members = np.arange(1, 30)
    z = philox.normals(5, philox.KIND_GA, 2, 4, members, D)
    got = gsm.children(elites, scale, 0.05, z, members, 1.0, 5, 2, 4)
    src = gsm.children(np.stack([np.zeros(D, np.float32), np.ones(D, np.float32)]), np.ones((2, D), np.float32), 0.0,
                       z, members, 1.0, 5, 2, 4).astype(np.int64)
    assert 0 < src.mean() < 1                                            # both elites contribute
    for r in range(len(members)):
        p = np.where(src[r] == 1, elites[1], elites[0])
        c = np.where(src[r] == 1, np.float32(4.0), np.float32(0.5))
        want = (p + ((np.float32(0.05) * z[r]).astype(np.float32) * c).astype(np.float32)).astype(np.float32)
        assert np.array_equal(got[r], want)


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200 import main
    return main.Args(main.parse_arguments(argv))


def test_flag_defaults_and_values():
    from coevonet_b200 import engine
    a = _cli(["--algorithm=GA", "--population=8"])
    assert (a.ga_safe_mutation, a.ga_safe_mutation_floor) == (False, None)
    assert engine.ga_safe_mutation(a) == {"ga_safe_mutation": False, "ga_safe_mutation_floor": None}
    a = _cli(["--algorithm=GA", "--population=8", "--ga_safe_mutation"])
    assert engine.ga_safe_mutation(a) == {"ga_safe_mutation": True, "ga_safe_mutation_floor": 0.01}
    a = _cli(["--algorithm=GA", "--population=8", "--ga_safe_mutation", "--ga_safe_mutation_floor=0.5"])
    assert engine.ga_safe_mutation(a) == {"ga_safe_mutation": True, "ga_safe_mutation_floor": 0.5}
    assert engine.ga_safe_mutation(types.SimpleNamespace(algorithm="GA")) == engine.GA_SAFE_MUTATION_DEFAULTS


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=ES", "--ga_safe_mutation"], "ES"),
    (["--algorithm=ES", "--ga_safe_mutation_floor=0.1"], "ES"),
    (["--algorithm=GA", "--ga_safe_mutation_floor=0.1"], "needs ga_safe_mutation"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=0"], "finite and > 0"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=-1"], "finite and > 0"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=nan"], "finite and > 0"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=inf"], "finite and > 0"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=1e300"], "finite and > 0"),
    (["--algorithm=GA", "--ga_safe_mutation", "--ga_safe_mutation_floor=1e-50"], "finite and > 0"),
])
def test_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_engines_refuse_bad_settings():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="ES"):
        engine.ESEngine(_args(4, algorithm="ES", ga_safe_mutation=True), "cpu", {}, kernels=_backend())
    with pytest.raises(ValueError, match="needs ga_safe_mutation"):
        _engine(4, ga_safe_mutation_floor=0.1)
    with pytest.raises(ValueError, match="finite"):
        _engine(4, ga_safe_mutation=True, ga_safe_mutation_floor=float("inf"))


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ga_safe_mutation_backend
    return ga_safe_mutation_backend


class _Log:
    """The checker backend, logging the name of every call the engine makes."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        fn = getattr(_backend(), name)
        if not callable(fn):
            return fn

        def logged(*a, **kw):
            self.calls.append((name, tuple(sorted(kw))))
            return fn(*a, **kw)
        return logged


def _args(P, record_history=True, **opts):
    a = types.SimpleNamespace(
        algorithm="GA", generations=8, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.04, mutation_power_adversary=0.03,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=1, reference_compat=True, init_states="device", seed=99, plots=False,
        record_history=record_history)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _rows(P, seed=700):
    from coevonet_b200 import layout
    pop, hof, founder = {}, {}, {}
    for i, r in enumerate(ROLES):
        in_dim = layout.OBS_DIM[r]
        rows = np.zeros((P + 3, layout.fc_pitch(in_dim)), dtype=np.float32)
        rows[:, :layout.fc_dim(in_dim)] = weights.make_fc_rows(P + 3, in_dim, seed + i, ln_jitter=0.02)
        pop[r] = torch.from_numpy(rows[:P].copy())
        hof[r] = torch.from_numpy(rows[P:P + 2].copy())
        founder[r] = torch.from_numpy(rows[P + 2].copy())
    return pop, hof, founder


def _engine(P, comm=None, kernels=None, **kw):
    from coevonet_b200 import engine
    pop, hof, founder = _rows(P)
    shard = engine.Shard(P, comm.rank if comm else 0, comm.world if comm else 1)
    sl = slice(shard.row0, shard.row0 + shard.n_local)
    return engine.GAEngine(_args(P, **kw), "cpu", {r: pop[r][sl].clone() for r in ROLES}, hof, founder,
                           kernels=kernels or _backend(), comm=comm)


def test_off_issues_the_default_calls():
    logs, states = [], []
    for kw in ({}, {"ga_safe_mutation": False}):
        log = _Log()
        eng = _engine(4, kernels=log, **kw)
        for _ in range(2):
            eng.step()
        assert eng.history[1]["safe_mutation_scale"] is None and eng.novelty_probe_obs is None
        logs.append(log.calls)
        states.append((eng.gstate.clone(), {r: eng.pop[r].clone() for r in ROLES}))
    assert logs[0] == logs[1]
    assert ("ga_repopulate", ("crossover_rate", "out")) in logs[0]
    assert not any("safe" in c[0] or "probe" in c[0] for c in logs[0])
    assert torch.equal(states[0][0], states[1][0])
    for r in ROLES:
        assert torch.equal(states[0][1][r], states[1][1][r])
    sd = eng.state_dict()
    assert sd["ga_safe_mutation"] == {"ga_safe_mutation": False, "ga_safe_mutation_floor": None}


SIGMA = {"agent_0": 0.05, "agent_1": 0.04, "adversary_0": 0.03}


@pytest.mark.parametrize("extra", [{}, {"crossover_rate": 0.5, "ga_novelty_weight": 0.5}], ids=["plain", "composed"])
def test_engine_follows_the_oracle(extra):
    """Every child of 3 generations is the oracle's formula on the engine's elites and their scale rows; the history
    statistics are those of the scale rows."""
    from coevonet_b200 import layout
    P, E = 6, 2
    eng = _engine(P, **SAFE, **extra)
    obs = {r: en.probe_obs(en.probe_states(99), r) for r in ROLES}
    for r in ROLES:
        assert np.array_equal(eng.novelty_probe_obs[r].numpy(), obs[r])
    rate = extra.get("crossover_rate", 0.0)
    for g in range(3):
        before = {r: eng.pop[r].numpy().copy() for r in ROLES}
        eng.step()
        h = eng.history[g]
        for r in ROLES:
            in_dim = layout.OBS_DIM[r]
            D = layout.fc_dim(in_dim)
            elites = before[r][h["elite_ids"][r]]
            scale = gsm.scale_rows(elites, in_dim, obs[r], SAFE["ga_safe_mutation_floor"])
            assert np.array_equal(eng.safe_scale[r].numpy(), scale), (g, r)
            members = np.arange(P)
            z = philox.normals(99, philox.KIND_GA, layout.ROLE_ID[r], g, members, D)
            want = gsm.children(elites[:, :D], scale, SIGMA[r], z, members, rate, 99, layout.ROLE_ID[r], g)
            assert np.array_equal(eng.pop[r].numpy()[:, :D], want), (g, r)
            assert not eng.pop[r].numpy()[:, D:].any()
            c = scale[:, :D]
            st = h["safe_mutation_scale"][r]
            assert st["min"] == float(c.min()) and st["max"] == float(c.max())
            assert st["mean"] == pytest.approx(float(c.astype(np.float64).mean()), rel=1e-12)
            assert st["n_floor"] == int((c == np.float32(1) / np.float32(0.05)).sum())


def test_safe_mutation_changes_the_children():
    a = _engine(5)
    b = _engine(5, **SAFE)
    a.step()
    b.step()
    for r in ROLES:
        assert np.array_equal(a.history[0]["elite_ids"][r], b.history[0]["elite_ids"][r])
        assert torch.equal(a.pop[r][0], b.pop[r][0])                       # row 0: the best, unmutated
        assert not torch.equal(a.pop[r][1:], b.pop[r][1:])


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(SAFE, record_history=False)
    full = _engine(5, **kw)
    for _ in range(3):
        full.step(sync=False)
    first = _engine(5, **kw)
    first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "safe.pt")
    second = _engine(5, **kw)
    second.load_state_dict(torch.load(tmp_path / "safe.pt", weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    for r in ROLES:
        assert torch.equal(second.pop[r], full.pop[r]) and torch.equal(second.hof[r], full.hof[r])


def test_resume_refuses_other_settings():
    safe = _engine(4, record_history=False, **SAFE)
    safe.step(sync=False)
    sd = safe.state_dict()
    assert sd["ga_safe_mutation"] == {"ga_safe_mutation": True, "ga_safe_mutation_floor": 0.05}
    with pytest.raises(ValueError, match="safe mutations"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="safe mutations"):
        _engine(4, record_history=False, ga_safe_mutation=True).load_state_dict(sd)
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    old = plain.state_dict()
    del old["ga_safe_mutation"]                 # written before the option existed: loads as off
    fresh = _engine(4, record_history=False)
    fresh.load_state_dict(old)
    for r in ROLES:
        assert torch.equal(fresh.pop[r], plain.pop[r])
    with pytest.raises(ValueError, match="safe mutations"):
        _engine(4, record_history=False, **SAFE).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **SAFE)
    evs = [eng.step() for _ in range(3)]
    q.put(dict(rank=rank, evs=np.asarray(evs), row0=eng.shard.row0, n_local=eng.shard.n_local,
               elite_ids=np.stack([eng.history[g]["elite_ids"][r] for g in range(3) for r in ROLES]),
               scale=np.concatenate([eng.safe_scale[r].numpy() for r in ROLES], axis=1),
               hof=np.concatenate([eng.hof[r].numpy() for r in ROLES], axis=1),
               pop=np.concatenate([eng.pop[r].numpy() for r in ROLES], axis=1)))
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
def test_safe_mutation_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows: every rank computes the same scale rows from the all-reduced elites."""
    P = 5
    single = _launch(1, P, 29691)[0]
    two = _launch(2, P, 29692)
    for o in two:
        for key in ("elite_ids", "scale", "hof"):
            assert np.array_equal(o[key], single[key]), key
        np.testing.assert_allclose(o["evs"], single["evs"], rtol=1e-12)
        sl = slice(o["row0"], o["row0"] + o["n_local"])
        assert np.array_equal(o["pop"], single["pop"][sl])


def test_safe_mutation_kernels_do_not_spill():
    """ptxas's report of the build: every kernel of ga_safe_mutation.cu without spills or a stack frame."""
    log = os.path.join(ROOT, "coevonet_b200", "csrc", "ga_safe_mutation.ptxas.log")
    if not os.path.isfile(log):
        pytest.skip("library not built")
    text = open(log).read()
    frames = [ln for ln in text.splitlines() if "stack frame" in ln]
    assert len(frames) == 8
    assert all(ln.strip() == "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" for ln in frames)
