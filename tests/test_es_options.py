"""The opt-in Co-ES update options (mirrored sampling, centered-rank fitness shaping, Adam / L2 apply) on the host:
the NumPy restatements the GPU tests check the kernels against, flag validation, and the engine's sharding /
checkpoint logic with the checker backend (tests/es_options_backend.py)."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy.stats import rankdata

from oracle import es_options as oes, layout as olayout, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
ALL_ON = dict(mirrored_sampling=True, fitness_shaping="centered_rank", es_optimizer="adam", learning_rate=0.01,
              l2_coeff=0.005)


# ---------------------------------------------------------------------------------------------------------------
# restatements
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [1, 2, 7, 1000])
def test_centered_ranks_match_rankdata(P):
    rng = np.random.default_rng(P)
    cases = [rng.normal(size=P), np.round(rng.normal(size=P), 1)]          # distinct values, many ties
    if P > 1:
        z = rng.normal(size=P)
        z[rng.random(P) < 0.3] = 0.0
        z[rng.random(P) < 0.3] = -0.0                                      # -0.0 == +0.0
        cases.append(z)
        n = np.round(rng.normal(size=P), 1)
        n[rng.random(P) < 0.2] = np.nan                                    # NaNs tie below every number
        n[0] = np.nan
        cases.append(n)
    for f in cases:
        got = oes.centered_ranks(f)
        want = rankdata(np.where(np.isnan(f), -np.inf, f), method="average") - 1.0
        want = want / (P - 1) - 0.5 if P > 1 else np.zeros(P)
        assert np.array_equal(got, want)
        assert got.dtype == np.float64 and np.all(np.abs(got) <= 0.5)
    assert oes.centered_ranks([-0.0, 0.0]).tolist() == [0.0, 0.0]
    assert oes.centered_ranks([np.nan, -np.inf, np.nan]).tolist() == [-0.25, 0.5, -0.25]


def _textbook_adam(theta, grads, lr, l2):
    """Adam in float64, as written in Kingma & Ba, ascending (theta += step)."""
    m = np.zeros_like(theta)
    v = np.zeros_like(theta)
    for t, gh in enumerate(grads, start=1):
        g = gh - l2 * theta
        m = 0.9 * m + 0.1 * g
        v = 0.999 * v + 0.001 * g * g
        theta = theta + lr * (m / (1 - 0.9 ** t)) / (np.sqrt(v / (1 - 0.999 ** t)) + 1e-8)
    return theta


def test_es_apply_restatement_follows_textbook_adam_and_keeps_layernorm_bits():
    from coevonet_b200 import layout
    in_dims = [10, 10, 8]
    rng = np.random.default_rng(5)
    mask = np.concatenate([np.isin(np.arange(layout.fc_pitch(d)), olayout.fc_perturbable_index(d)) for d in in_dims])
    n = mask.size
    theta0 = rng.normal(0, 0.1, n).astype(np.float32)
    theta0[~mask] = rng.normal(1, 0.02, (~mask).sum()).astype(np.float32)
    # |g| bounded away from 0: there Adam's step is ~ lr * sign(g), and a rounding that flips the sign of a g ~ 0
    # (in either computation) would move theta by ~lr
    sign = rng.choice([-1.0, 1.0], n)
    grads = [(sign * rng.uniform(0.1, 0.5, n)).astype(np.float32) for _ in range(4)]
    lr, l2 = 0.01, 0.005
    theta, m, v = theta0, np.full(n, -7.0, np.float32), np.full(n, 3.0, np.float32)
    m[mask] = 0
    v[mask] = 0
    m0, v0 = m.copy(), v.copy()
    for t, g in enumerate(grads, start=1):
        theta, m, v = oes.es_apply(theta, g, mask, "adam", lr, l2, t, m, v)
    want = _textbook_adam(theta0[mask].astype(np.float64), [g[mask].astype(np.float64) for g in grads], lr, l2)
    # four steps of size ~lr: a few fp32 roundings (ulp(0.5) = 6e-8) from the fp64 value
    np.testing.assert_allclose(theta[mask], want, rtol=0, atol=5e-7)
    assert np.array_equal(theta[~mask].view(np.uint32), theta0[~mask].view(np.uint32))
    assert np.array_equal(m[~mask], m0[~mask]) and np.array_equal(v[~mask], v0[~mask])
    # sgd + l2: theta += lr * (g - l2 theta)
    th, _, _ = oes.es_apply(theta0, grads[0], mask, "sgd", 0.1, l2)
    want = theta0[mask].astype(np.float64) + 0.1 * (grads[0][mask] - l2 * theta0[mask].astype(np.float64))
    np.testing.assert_allclose(th[mask], want, rtol=0, atol=1e-7)
    assert np.array_equal(th[~mask].view(np.uint32), theta0[~mask].view(np.uint32))


def test_es_apply_step_size_is_adams_bias_correction():
    for t in (1, 2, 10, 1000):
        a = np.float32(0.01 * math.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t))
        g = np.full(1, 0.25, np.float32)
        m = np.full(1, 0.5, np.float32)
        v = np.full(1, 0.0625, np.float32)
        th, m2, v2 = oes.es_apply(np.zeros(1, np.float32), g, [True], "adam", 0.01, 0.0, t, m, v)
        want = (a * m2[0]) / (np.sqrt(v2[0]) + np.float32(1e-8))
        assert th[0] == want


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_flag_defaults_and_parsing():
    a = _cli(["--algorithm=ES"])
    assert (a.mirrored_sampling, a.fitness_shaping, a.es_optimizer, a.l2_coeff) == (False, "none", "sgd", 0.0)
    a = _cli(["--algorithm=ES", "--population=8", "--mirrored_sampling", "--fitness_shaping=centered_rank",
              "--es_optimizer=adam", "--learning_rate=0.01", "--l2_coeff=0.005"])
    from coevonet_b200.engine import es_options
    assert es_options(a) == {"mirrored_sampling": True, "fitness_shaping": "centered_rank", "es_optimizer": "adam",
                             "l2_coeff": 0.005}
    with pytest.raises(SystemExit):
        _cli(["--algorithm=ES", "--es_optimizer=rmsprop"])


def test_mirrored_sampling_needs_an_even_population():
    with pytest.raises(ValueError, match="even population"):
        _cli(["--algorithm=ES", "--population=7", "--mirrored_sampling"])
    _cli(["--algorithm=ES", "--population=8", "--mirrored_sampling"])


@pytest.mark.parametrize("flag", ["--mirrored_sampling", "--fitness_shaping=centered_rank", "--es_optimizer=adam",
                                  "--l2_coeff=0.01"])
def test_es_options_are_refused_with_ga(flag):
    with pytest.raises(ValueError, match="GA"):
        _cli(["--algorithm=GA", "--population=8", flag])
    _cli(["--algorithm=ES", "--population=8", flag])


def test_ga_engine_refuses_es_options():
    eng_args = _args(4, mirrored_sampling=True)
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="GA"):
        engine.GAEngine(eng_args, "cpu", {}, {}, {}, kernels=_backend())


# ---------------------------------------------------------------------------------------------------------------
# engines on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import es_options_backend
    return es_options_backend


def _args(P, record_history=True, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=4, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
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


def _engine(P, comm=None, **kw):
    from coevonet_b200 import engine
    return engine.ESEngine(_args(P, **kw), "cpu", _theta(), kernels=_backend(), comm=comm)


def test_engine_without_the_new_attributes_equals_defaults():
    plain = _engine(4)
    explicit = _engine(4, mirrored_sampling=False, fitness_shaping="none", es_optimizer="sgd", l2_coeff=0.0)
    assert plain.options == explicit.options and not plain.fused_apply and plain.adam_m is None
    for _ in range(2):
        assert plain.step() == explicit.step()
    assert torch.equal(plain.theta_cat, explicit.theta_cat)
    for h0, h1 in zip(plain.history, explicit.history):
        for r in ROLES:
            assert np.array_equal(h0["rewards"][r], h1["rewards"][r])
            assert np.array_equal(h0["delta"][r], h1["delta"][r])
            assert h0["shaped_fitness"][r] is None and h1["shaped_fitness"][r] is None
    assert "adam_m" not in plain.state_dict() and plain.state_dict()["es_options"] == plain.options


def test_mirrored_members_are_antithetic_pairs():
    from coevonet_b200 import layout
    eng = _engine(6, **ALL_ON)
    eng.evaluate()
    for r in ROLES:
        in_dim = layout.OBS_DIM[r]
        D = layout.fc_dim(in_dim)
        pidx = olayout.fc_perturbable_index(in_dim)
        theta = eng.theta[r].numpy()[:D]
        z = philox.normals(99, oes.KIND_ES_MIRROR, philox.ROLE_ID[r], 0, np.arange(3), D)
        d = (np.float32(0.05) * z[:, pidx]).astype(np.float32)
        mem = eng.members[r].numpy()
        for q in range(3):
            assert np.array_equal(mem[2 * q, pidx], (theta[pidx] + d[q]).astype(np.float32))
            assert np.array_equal(mem[2 * q + 1, pidx], (theta[pidx] + (-d[q])).astype(np.float32))
        ln = np.setdiff1d(np.arange(D), pidx)
        assert np.all(mem[:, ln] == theta[ln])
    # the engine records the shaped global fitness: ranks of the (shared) fitness
    eng.update()
    for r in ROLES:
        assert np.array_equal(eng.shaped_fitness[r].numpy(), oes.centered_ranks(eng.fitness[r].numpy()))


@pytest.mark.parametrize("regenerate", [False, True])
def test_resume_with_all_options_equals_uninterrupted_run(tmp_path, regenerate):
    kw = dict(ALL_ON, record_history=False, update_from_members=not regenerate)
    full = _engine(4, **kw)
    for _ in range(4):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    path = tmp_path / "es.pt"
    torch.save(first.state_dict(), path)
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(path, weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.theta_cat, full.theta_cat)
    assert torch.equal(second.adam_m, full.adam_m) and torch.equal(second.adam_v, full.adam_v)
    assert float(full.adam_v.abs().max()) > 0


def test_resume_refuses_other_options(tmp_path):
    on = _engine(4, record_history=False, **ALL_ON)
    on.step(sync=False)
    sd = on.state_dict()
    with pytest.raises(ValueError, match="ES options"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="ES options"):
        _engine(4, record_history=False, **dict(ALL_ON, l2_coeff=0.0)).load_state_dict(sd)
    # a checkpoint without es_options (written before they existed) loads into a default run only
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    old = plain.state_dict()
    del old["es_options"]
    _engine(4, record_history=False).load_state_dict(old)
    with pytest.raises(ValueError, match="ES options"):
        _engine(4, record_history=False, **ALL_ON).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **ALL_ON)
    evs = [eng.step() for _ in range(2)]
    q.put(dict(rank=rank, evs=np.asarray(evs),
               rewards=np.stack([eng.history[g]["rewards"][r] for g in range(2) for r in ROLES]),
               shaped=np.stack([eng.history[g]["shaped_fitness"][r] for g in range(2) for r in ROLES]),
               theta=np.stack([eng.theta[r].numpy()[:5000] for r in ROLES]),
               m=eng.adam_m.numpy()[:5000].copy(), v=eng.adam_v.numpy()[:5000].copy()))
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
def test_es_options_two_ranks_match_one_rank():
    """P = 6 over two ranks is 3 + 3 rows: the pair (2, 3) is cut by the shard boundary."""
    P = 6
    single = _launch(1, P, 29631)[0]
    two = _launch(2, P, 29632)
    for o in two:
        np.testing.assert_allclose(o["rewards"], single["rewards"], rtol=1e-12, atol=0)
        assert np.array_equal(o["shaped"], single["shaped"])          # ranks of the gathered global fitness
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
    for k in ("theta", "m", "v"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree
