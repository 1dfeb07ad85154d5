"""Separable NES (a per-parameter mutation strength) on the host: the NumPy restatement against a textbook fp64 SNES
step, the default sigma learning rate, flag validation, and the ES engine's separable path with the checker backend
(tests/snes_backend.py): members, mirrored pairs, clamps, resume, checkpoint settings and two gloo ranks."""
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_options as oes, ga_es, layout as olayout, philox, snes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SNES = dict(es_distribution="separable", learning_rate=1.0)
SNES_ALL = dict(SNES, mirrored_sampling=True, fitness_shaping="centered_rank")


# ---------------------------------------------------------------------------------------------------------------
# restatement
# ---------------------------------------------------------------------------------------------------------------
def test_restatement_follows_a_textbook_snes_step():
    rng = np.random.default_rng(1)
    n, d = 64, 3000
    theta = rng.normal(0, 0.2, d).astype(np.float32)
    sigma = rng.uniform(0.02, 0.08, d).astype(np.float32)
    z = rng.normal(size=(n, d)).astype(np.float32)
    F = rng.normal(-20, 5, n)
    lr, eta = 1.0, 0.05
    mask = np.ones(d, bool)
    rows, noise = snes.perturb(theta, sigma, z, np.arange(d))
    np.testing.assert_allclose(rows, theta.astype(np.float64) + sigma.astype(np.float64) * z, rtol=0, atol=1e-7)
    gm, gs = snes.gradients(noise, F, n)
    th, sg = snes.apply(theta, sigma, gm, gs, mask, lr, eta, 1e-6, 10.0)
    # Wierstra et al. 2014, Algorithm 6 (SNES) in fp64: utilities F, s_k = z_k
    z64, F32 = z.astype(np.float64), F.astype(np.float32).astype(np.float64)
    gm64 = z64.T @ F32 / n
    gs64 = (z64 * z64 - 1).T @ F32 / n
    th64 = theta + lr * sigma.astype(np.float64) * gm64
    sg64 = sigma * np.exp(eta / 2 * gs64)
    # fp32 sums of 64 terms of size ~20: a few ulp of the sum
    np.testing.assert_allclose(gm, gm64, rtol=0, atol=2e-4 * np.abs(gm64).max())
    np.testing.assert_allclose(gs, gs64, rtol=0, atol=2e-4 * np.abs(gs64).max())
    np.testing.assert_allclose(th, th64, rtol=0, atol=1e-5 * np.abs(th64).max())
    np.testing.assert_allclose(sg, sg64, rtol=1e-5, atol=0)
    assert not np.array_equal(sg, sigma)
    # the clamps
    _, sg = snes.apply(theta, sigma, gm, gs, mask, lr, 2.0, 0.03, 0.07)
    assert sg.min() == np.float32(0.03) and sg.max() == np.float32(0.07)


def test_restatement_with_a_constant_sigma_is_the_isotropic_perturbation():
    in_dim = 10
    D = olayout.fc_dim(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    theta = np.random.default_rng(2).normal(0, 0.1, D).astype(np.float32)
    sigma = np.zeros(D, np.float32)
    sigma[pidx] = np.float32(0.05)
    z = philox.normals(5, philox.KIND_ES, 0, 3, np.arange(7, 12), D)
    rows, _ = snes.perturb(theta, sigma, z, pidx)
    assert np.array_equal(rows, ga_es.es_perturb(theta, 0.05, z, pidx)[0])
    zq = philox.normals(5, oes.KIND_ES_MIRROR, 0, 3, np.arange(3, 6), D)        # pairs of members 7 .. 11
    rows, _ = snes.perturb(theta, sigma, zq[(np.arange(7, 12) >> 1) - 3], pidx, 7, mirrored=True)
    assert np.array_equal(rows, oes.es_perturb_mirrored(theta, 0.05, zq, pidx, 7, 5)[0])


def test_default_sigma_learning_rate_per_role():
    from coevonet_b200 import engine, layout
    eng = _engine(4, **SNES)
    for r in ROLES:
        d = len(olayout.fc_perturbable_index(layout.OBS_DIM[r]))
        want = (3 + np.log(d)) / (5 * np.sqrt(d))
        assert eng.sigma_lr[r] == want == snes.default_sigma_lr(d) == engine.default_sigma_learning_rate(d)
        assert 0.007 < want < 0.009                                        # d ~ 1.4e5
    assert eng.sigma_lr["agent_0"] == eng.sigma_lr["agent_1"] != eng.sigma_lr["adversary_0"]
    eng = _engine(4, sigma_learning_rate=0.02, **SNES)
    assert all(eng.sigma_lr[r] == 0.02 for r in ROLES)


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_distribution_flags_defaults_and_parsing():
    from coevonet_b200.engine import ES_DISTRIBUTION_DEFAULTS, es_distribution
    a = _cli(["--algorithm=ES"])
    assert (a.es_distribution, a.sigma_learning_rate) == ("isotropic", None)
    assert es_distribution(a) == ES_DISTRIBUTION_DEFAULTS
    assert es_distribution(types.SimpleNamespace(population=4)) == ES_DISTRIBUTION_DEFAULTS    # attributes absent
    a = _cli(["--algorithm=ES", "--population=8", "--es_distribution=separable", "--mirrored_sampling",
              "--fitness_shaping=centered_rank", "--learning_rate=1.0", "--sigma_learning_rate=0.01"])
    assert es_distribution(a) == {"es_distribution": "separable", "sigma_learning_rate": 0.01}
    with pytest.raises(SystemExit):
        _cli(["--algorithm=ES", "--es_distribution=cma"])
    with pytest.raises(ValueError, match="isotropic"):
        es_distribution(types.SimpleNamespace(es_distribution="cma"))


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=GA", "--es_distribution=separable"], "GA"),
    (["--algorithm=GA", "--sigma_learning_rate=0.01"], "GA"),
    (["--algorithm=ES", "--es_distribution=separable", "--es_optimizer=adam"], "adam"),
    (["--algorithm=ES", "--es_distribution=separable", "--l2_coeff=0.01"], "l2_coeff"),
    (["--algorithm=ES", "--es_distribution=separable", "--adaptive"], "adaptive"),
    (["--algorithm=ES", "--es_distribution=separable", "--sigma_learning_rate=0"], "> 0"),
    (["--algorithm=ES", "--es_distribution=separable", "--sigma_learning_rate=-0.1"], "> 0"),
    (["--algorithm=ES", "--es_distribution=separable", "--sigma_learning_rate=nan"], "> 0"),
    (["--algorithm=ES", "--sigma_learning_rate=0.01"], "separable"),
    (["--algorithm=ES", "--es_distribution=isotropic", "--sigma_learning_rate=0.01"], "separable"),
])
def test_distribution_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_ga_engine_refuses_the_separable_distribution():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="GA"):
        engine.GAEngine(_args(4, algorithm="GA", es_distribution="separable"), "cpu", {}, {}, {}, kernels=_backend())


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import snes_backend
    return snes_backend


def _args(P, record_history=True, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=4, population=P, hof_size=2, game="simple_adversary_v3",
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


def _engine(P, comm=None, **kw):
    from coevonet_b200 import engine
    return engine.ESEngine(_args(P, **kw), "cpu", _theta(), kernels=_backend(), comm=comm)


def _masks(in_dim):
    from coevonet_b200 import layout
    pitch = layout.fc_pitch(in_dim)
    pert = np.zeros(pitch, bool)
    pert[olayout.fc_perturbable_index(in_dim)] = True
    return pert


def test_initial_sigma_row_and_isotropic_engine_state():
    from coevonet_b200 import layout
    eng = _engine(4, **SNES)
    for r, s0 in zip(ROLES, (0.05, 0.04, 0.03)):
        s = eng.sigma_rows[r].numpy()
        pert = _masks(layout.OBS_DIM[r])
        assert np.all(s[pert] == np.float32(s0)) and np.all(s[~pert].view(np.uint32) == 0)
    iso = _engine(4)
    assert not iso.separable and iso.sigma_cat is None and iso.grad_cat is None
    iso.step()
    assert all(iso.history[0]["sigma_stats"][r] is None for r in ROLES)
    assert "sigma" not in iso.state_dict() and iso.state_dict()["es_distribution"] == iso.distribution


@pytest.mark.parametrize("mirrored", [False, True])
def test_members_are_mu_plus_sigma_times_the_philox_normals(mirrored):
    from coevonet_b200 import layout
    eng = _engine(6, mirrored_sampling=mirrored, **SNES)
    eng.step()                                    # sigma is no longer uniform
    h = eng.history[0]
    sigma = {r: eng.sigma_rows[r].numpy().copy() for r in ROLES}
    for r in ROLES:
        st = h["sigma_stats"][r]
        pidx = olayout.fc_perturbable_index(layout.OBS_DIM[r])
        s = sigma[r][pidx]
        np.testing.assert_allclose(st, (s.mean(), s.min(), s.max(), s.std()), rtol=1e-5)
        assert st[1] < st[2]
    eng.evaluate()
    for r in ROLES:
        in_dim = layout.OBS_DIM[r]
        D = layout.fc_dim(in_dim)
        pidx = olayout.fc_perturbable_index(in_dim)
        mu = eng.theta[r].numpy()[:D]
        mem = eng.members[r].numpy()
        if mirrored:
            z = philox.normals(99, oes.KIND_ES_MIRROR, philox.ROLE_ID[r], 1, np.arange(3), D)[:, pidx]
            for q in range(3):
                d = (sigma[r][pidx] * z[q]).astype(np.float32)
                assert np.array_equal(mem[2 * q, pidx], (mu[pidx] + d).astype(np.float32))
                assert np.array_equal(mem[2 * q + 1, pidx], (mu[pidx] + (-d)).astype(np.float32))
        else:
            z = philox.normals(99, philox.KIND_ES, philox.ROLE_ID[r], 1, np.arange(6), D)[:, pidx]
            want = (mu[pidx] + (sigma[r][pidx] * z).astype(np.float32)).astype(np.float32)
            assert np.array_equal(mem[:, pidx], want)
        ln = np.setdiff1d(np.arange(D), pidx)
        assert np.all(mem[:, ln] == mu[ln]) and np.all(mem[:, D:] == 0)


def test_sigma_moves_inside_the_clamps_and_layernorm_bits_stay():
    from coevonet_b200 import layout
    kw = dict(SNES_ALL, sigma_learning_rate=20.0, min_mutation_power=0.035, max_mutation_power=0.045)
    eng = _engine(6, **kw)
    theta0 = eng.theta_cat.numpy().copy()
    for _ in range(2):
        eng.step()
    sig = eng.sigma_cat.numpy()
    th = eng.theta_cat.numpy()
    pert = np.concatenate([_masks(layout.OBS_DIM[r]) for r in ROLES])
    assert np.array_equal(th[~pert].view(np.uint32), theta0[~pert].view(np.uint32))
    assert np.all(sig[~pert].view(np.uint32) == 0)
    s = sig[pert]
    assert s.min() == np.float32(0.035) and s.max() == np.float32(0.045)          # both clamps reached
    inside = s[(s > np.float32(0.035)) & (s < np.float32(0.045))]
    assert inside.size > 0 and np.unique(inside).size > 10
    assert np.any(th[pert] != theta0[pert])
    # the recorded delta is g_mu (the engine's ascent estimate), the same for every rank
    assert np.array_equal(np.concatenate([eng.history[-1]["delta"][r] for r in ROLES]),
                          eng.grad_cat.numpy()[:th.size])


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(SNES_ALL, record_history=False)
    full = _engine(4, **kw)
    for _ in range(4):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "snes.pt")
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(tmp_path / "snes.pt", weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.theta_cat, full.theta_cat)
    assert torch.equal(second.sigma_cat, full.sigma_cat)
    assert not torch.equal(full.sigma_cat, _engine(4, **kw).sigma_cat)


def test_resume_refuses_other_distribution_settings():
    sep = _engine(4, record_history=False, **SNES)
    sep.step(sync=False)
    sd = sep.state_dict()
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False, sigma_learning_rate=0.01, **SNES).load_state_dict(sd)
    iso = _engine(4, record_history=False)
    iso.step(sync=False)
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False, **SNES).load_state_dict(iso.state_dict())
    # a checkpoint without the settings (written before they existed) is isotropic
    old = iso.state_dict()
    del old["es_distribution"]
    _engine(4, record_history=False).load_state_dict(old)
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False, **SNES).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **SNES_ALL)
    evs = [eng.step() for _ in range(2)]
    q.put(dict(rank=rank, evs=np.asarray(evs),
               rewards=np.stack([eng.history[g]["rewards"][r] for g in range(2) for r in ROLES]),
               shaped=np.stack([eng.history[g]["shaped_fitness"][r] for g in range(2) for r in ROLES]),
               theta=eng.theta_cat.numpy().copy(), sigma=eng.sigma_cat.numpy().copy()))
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
def test_separable_two_ranks_match_one_rank():
    """P = 6 over two ranks is 3 + 3 rows: the pair (2, 3) is cut by the shard boundary."""
    P = 6
    single = _launch(1, P, 29641)[0]
    two = _launch(2, P, 29642)
    for o in two:
        np.testing.assert_allclose(o["rewards"], single["rewards"], rtol=1e-12, atol=0)
        assert np.array_equal(o["shaped"], single["shaped"])
        # the two ranks' partial sums are added in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["sigma"], single["sigma"], rtol=1e-5, atol=0)
    for k in ("theta", "sigma"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree
