"""Co-ES novelty search on the GPU: the probe-observation kernel bit for bit against the oracle, the behaviour
characterisation kernel against the oracle's fp32 forward (P = 1, 1,024 and 2 n_sm + 3, row-strided members with NaN
padding) and bit for bit against chunked launches of one job per CTA, the k-NN kernel bit for bit against the oracle,
and the engine: w = 0 against the default, w = 1 and 0.5 against the oracle's fitness, determinism, resume, the other
Co-ES options, and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_novelty as en, es_options as oes, philox

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 4242
#: largest |kernel - oracle| of a characterisation entry (a probability) allowed; the fp32 forwards sum in other
#: orders, which moves the logits by a few ulps (profiles/r07_es_novelty_bc_error.json records the measured error,
#: written by tests/tools/novelty_bc_err.py)
BC_TOL = 2e-6


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _members(role, P, seed=SEED):
    """P sigma-0.05 members around a default-initialised base agent, fp32 [P, pitch] on the GPU."""
    from coevonet_b200 import layout, ops
    in_dim = layout.OBS_DIM[role]
    theta = ops.fc_init(in_dim, seed, role, 0, 1, "cuda")[0]
    return ops.es_perturb(theta, in_dim, 0.05, seed, role, 0, 0, P)


def _probe_obs(role, seed=SEED):
    from coevonet_b200 import ops
    states = ops.init_states(seed, en.PROBE_TAG, en.PROBES, "cuda")
    return ops.novelty_probe_obs(states, role)


def _oracle_bc(rows, role, obs):
    from coevonet_b200 import layout
    in_dim = layout.OBS_DIM[role]
    return en.bc(rows.cpu().numpy()[:, :layout.fc_dim(in_dim)], in_dim, obs.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------------
# probe observations
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("role", ROLES)
def test_probe_obs_kernel_is_bit_exact(role):
    from coevonet_b200 import ops
    states = ops.init_states(SEED, en.PROBE_TAG, en.PROBES, "cuda")
    assert np.array_equal(states.cpu().numpy(), en.probe_states(SEED))
    assert np.array_equal(ops.novelty_probe_obs(states, role).cpu().numpy(), en.probe_obs(en.probe_states(SEED), role))
    many = ops.init_states(SEED, 7, 1000, "cuda")
    assert np.array_equal(ops.novelty_probe_obs(many, role).cpu().numpy(),
                          en.probe_obs(philox.init_states(SEED, 7, 1000), role))


# ---------------------------------------------------------------------------------------------------------------
# behaviour characterisation
# ---------------------------------------------------------------------------------------------------------------
def _chunked(rows, in_dim, obs, chunk):
    """Launches of `chunk` rows each: with chunk <= n_sm every CTA runs one job."""
    from coevonet_b200 import ops
    return torch.cat([ops.novelty_bc(rows[i:i + chunk], in_dim, obs) for i in range(0, rows.shape[0], chunk)])


@pytest.mark.parametrize("role", ["agent_0", "adversary_0"])
@pytest.mark.parametrize("P", [1, 1024, "2sm+3"])
def test_bc_kernel_matches_the_oracle(role, P):
    from coevonet_b200 import layout, ops
    P = 2 * _n_sm() + 3 if P == "2sm+3" else P
    in_dim = layout.OBS_DIM[role]
    rows, obs = _members(role, P), _probe_obs(role)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    bc = ops.novelty_bc(rows, in_dim, obs, status=status)
    assert int(status.item()) == 0
    got = bc.cpu().numpy()
    want = _oracle_bc(rows, role, obs)
    err = np.abs(got - want).max()
    assert err <= BC_TOL, err
    np.testing.assert_allclose(got.reshape(P, 32, 5).sum(axis=2), 1.0, atol=1e-6)
    # every row bit for bit as in launches where each CTA runs one job, and again on a second run
    assert torch.equal(bc, _chunked(rows, in_dim, obs, _n_sm()))
    assert torch.equal(bc, ops.novelty_bc(rows, in_dim, obs))


def test_bc_kernel_row_strided_members_with_nan_padding():
    from coevonet_b200 import layout, ops
    role = "agent_1"
    in_dim = layout.OBS_DIM[role]
    P, D, pitch = 2 * _n_sm() + 3, layout.fc_dim(in_dim), layout.fc_pitch(in_dim)
    rows, obs = _members(role, P), _probe_obs(role)
    wide = torch.full((P, pitch + 32), float("nan"), device="cuda")
    wide[:, :D] = rows[:, :D]                              # NaN in the row padding and in the 32 extra floats
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    got = ops.novelty_bc(wide[:, :pitch], in_dim, obs, status=status)
    assert int(status.item()) == 0
    assert torch.equal(got, ops.novelty_bc(rows, in_dim, obs))
    # the output may be rows of a wider buffer too (a slot of the archive ring)
    ring = torch.full((P + 4, 160), -1.0, device="cuda")
    ops.novelty_bc(wide[:, :pitch], in_dim, obs, out=ring[2:P + 2])
    assert torch.equal(ring[2:P + 2], got) and bool((ring[:2] == -1).all()) and bool((ring[P + 2:] == -1).all())


def test_bc_kernel_flags_non_finite_logits():
    from coevonet_b200 import layout, ops
    role = "agent_0"
    in_dim = layout.OBS_DIM[role]
    rows, obs = _members(role, 8), _probe_obs(role)
    o = layout.fc_segments(in_dim)[0][4][1]                # fc2.weight
    rows[5, o + 3] = float("inf")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.novelty_bc(rows, in_dim, obs, status=status)
    assert int(status.item()) == 1
    with pytest.raises(ValueError):
        ops.raise_on_status(status)


def test_bc_wrapper_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    rows, obs = _members("agent_0", 4), _probe_obs("agent_0")
    with pytest.raises(_lib.CevError):
        ops.novelty_bc(rows.cpu(), 10, obs)
    with pytest.raises(_lib.CevError):
        ops.novelty_bc(rows, 10, obs[:16])
    with pytest.raises(_lib.CevError):
        ops.novelty_bc(rows[:, :100], 10, obs)
    with pytest.raises(_lib.CevError):
        ops.novelty_bc(rows, 10, obs, out=torch.empty((4, 150), device="cuda"))
    assert ops.novelty_bc(rows[:0], 10, obs).shape == (0, 160)


# ---------------------------------------------------------------------------------------------------------------
# k-NN novelty
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("filled,k", [(1, 1), (1, 10), (7, 10), (300, 10), (4096, 32), (4096, 1)])
def test_knn_kernel_is_bit_exact_on_kernel_characterisations(filled, k):
    from coevonet_b200 import ops
    role = "agent_0"
    obs = _probe_obs(role)
    bc = ops.novelty_bc(_members(role, 300), 10, obs)
    ring = ops.novelty_bc(_members(role, 4096, seed=SEED + 1), 10, obs)
    got = ops.novelty_knn(bc, ring, filled, k).cpu().numpy()
    want = en.novelty(bc.cpu().numpy(), ring[:filled].cpu().numpy(), k)
    assert np.array_equal(got, want)


def test_knn_kernel_is_bit_exact_on_ties():
    from coevonet_b200 import ops
    rng = np.random.default_rng(9)
    base = rng.dirichlet(np.ones(5), size=(40, 32)).reshape(40, 160).astype(np.float32)
    ring = np.concatenate([base, base, base[::-1], base[:5]])          # every entry two or three times
    bcs = np.concatenate([base[:20], base[:3] + np.float32(1e-3)])
    tb, tr = torch.from_numpy(bcs).cuda(), torch.from_numpy(ring).cuda()
    for filled in (1, 3, 40, 45, 80, len(ring)):
        for k in (1, 2, 3, 7, 32):
            got = ops.novelty_knn(tb, tr, filled, k).cpu().numpy()
            assert np.array_equal(got, en.novelty(bcs, ring[:filled], k)), (filled, k)
    assert float(ops.novelty_knn(tb[:1], tr, len(ring), 3)[0]) == 0.0


def test_knn_wrapper_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    bc, ring = torch.zeros((4, 160), device="cuda"), torch.zeros((8, 160), device="cuda")
    for filled, k in ((0, 1), (9, 1), (4, 0), (4, 33)):
        with pytest.raises(_lib.CevError):
            ops.novelty_knn(bc, ring, filled, k)
    with pytest.raises(_lib.CevError):
        ops.novelty_knn(bc.cpu(), ring.cpu(), 4, 2)
    with pytest.raises(_lib.CevError):
        ops.novelty_knn(bc[:, :100].contiguous(), ring, 4, 2)


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


def _engine(P, **opts):
    from coevonet_b200 import engine, layout, ops
    theta = {r: ops.fc_init(layout.OBS_DIM[r], 5, r, 0, 1, "cuda")[0].cpu() for r in ROLES}
    return engine.ESEngine(_args(P, **opts), torch.device("cuda", 0), theta)


NOV = dict(es_novelty_weight=0.5, es_novelty_k=4, es_novelty_archive=3, fitness_shaping="centered_rank")


def _bits(eng):
    eng.check_status()
    out = {"theta": eng.theta_cat.cpu().numpy().view(np.uint32), "gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["rew_" + r] = eng.rewards[r].cpu().numpy()
        if eng.novelty_w:
            out["nov_" + r] = eng.novelty[r].cpu().numpy()
            out["F_" + r] = eng.shaped_fitness[r].cpu().numpy()
    if eng.novelty_ring is not None:
        out["ring"] = eng.novelty_ring.cpu().numpy().view(np.uint32)
    return out


def _same(a, b, keys=None):
    for k in keys or a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("shaping", ["none", "centered_rank"])
def test_zero_weight_equals_the_default_engine(shaping):
    plain = _engine(64, fitness_shaping=shaping)
    off = _engine(64, fitness_shaping=shaping, es_novelty_weight=0.0)
    for _ in range(3):
        plain.step(sync=False)
        off.step(sync=False)
        _same(_bits(plain), _bits(off))
    assert off.novelty_ring is None


@pytest.mark.parametrize("w", [1.0, 0.5], ids=["ns", "nsr"])
def test_generations_match_the_oracle(w):
    """P = 32 over A + 1 generations: the novelty is the oracle's k-NN of the kernel's characterisations against the
    ring as it stood, F is the oracle's combination of the global ranks, the ring holds the base agents'
    characterisations, and those are the oracle's forward within BC_TOL."""
    from coevonet_b200 import layout, ops
    A, k = 3, 4
    eng = _engine(32, record_history=True, es_novelty_weight=w, es_novelty_k=k, es_novelty_archive=A,
                  fitness_shaping="centered_rank")
    obs = {r: _probe_obs(r) for r in ROLES}
    for r in ROLES:
        assert np.array_equal(eng.novelty_probe_obs[r].cpu().numpy(), en.probe_obs(en.probe_states(SEED), r))
    for g in range(A + 1):
        ring_before = eng.novelty_ring.cpu().numpy().copy()
        filled = eng.novelty_filled
        eng.step()
        h = eng.history[g]
        assert h["novelty_filled"] == filled
        for i, r in enumerate(ROLES):
            in_dim = layout.OBS_DIM[r]
            bc = ops.novelty_bc(eng.members[r], in_dim, obs[r])
            assert np.abs(bc.cpu().numpy() - _oracle_bc(eng.members[r], r, obs[r])).max() <= BC_TOL
            nov = en.novelty(bc.cpu().numpy(), ring_before[i, :filled], k)
            assert np.array_equal(h["novelty"][r], nov), (g, r)
            F = en.combine(oes.centered_ranks(eng.fitness[r].cpu().numpy()), oes.centered_ranks(nov), w)
            assert np.array_equal(h["shaped_fitness"][r], F), (g, r)
            slot = (eng.novelty_head - 1) % A
            assert torch.equal(eng.novelty_ring[i, slot], ops.novelty_bc(eng.theta[r].reshape(1, -1), in_dim, obs[r])[0])
    assert eng.novelty_filled == A


def test_deterministic_and_resume_is_bit_identical():
    a, b = _engine(64, **NOV), _engine(64, **NOV)
    for _ in range(2):
        a.step(sync=False)
        b.step(sync=False)
    _same(_bits(a), _bits(b))
    sd = a.state_dict()
    for _ in range(2):
        a.step(sync=False)
    c = _engine(64, **NOV)
    c.load_state_dict(sd)
    for _ in range(2):
        c.step(sync=False)
    _same(_bits(a), _bits(c))
    assert (a.novelty_head, a.novelty_filled) == (c.novelty_head, c.novelty_filled)


@pytest.mark.parametrize("opts", [dict(mirrored_sampling=True), dict(es_distribution="separable"),
                                  dict(es_subspace_dim=2), dict(es_hof_size=3, es_hof_opponents=2)],
                         ids=["mirrored", "separable", "subspace", "hof"])
def test_composes_with_the_other_options(opts):
    eng = _engine(64, **dict(NOV, **opts))
    eng.step(sync=False)
    eng.check_status()
    for r in ROLES:
        F = eng.shaped_fitness[r].cpu().numpy()
        assert F.shape == (64,) and np.all(np.isfinite(F))
        assert np.all(np.isfinite(eng.novelty[r].cpu().numpy()))
    assert np.all(np.isfinite(eng.theta_cat.cpu().numpy()))


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
    eng = engine.ESEngine(_args(P, E, **NOV), dev, theta, comm=comm)
    ring0 = eng.novelty_ring.cpu().numpy()
    eng.step(sync=False)
    first = dict(nov=np.stack([eng.novelty[r].cpu().numpy() for r in ROLES]),
                 F=np.stack([comm.all_gather_rows(eng.shaped_fitness[r], eng.shard).cpu().numpy() for r in ROLES]))
    eng.step(sync=False)
    eng.check_status()
    q.put((rank, dict(ring0=ring0, ring=eng.novelty_ring.cpu().numpy(), theta=eng.theta_cat.cpu().numpy(), **first)))
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
def test_novelty_sharded_over_two_gpus_equal_one_gpu():
    P, E = 387, 4                                  # 194 + 193 rows
    one = _launch(1, P, E, 29741)[0]
    two = _launch(2, P, E, 29742)
    assert np.array_equal(two[0]["ring"], two[1]["ring"]) and np.array_equal(two[0]["theta"], two[1]["theta"])
    for o in two:
        assert np.array_equal(o["ring0"], one["ring0"])
        assert np.array_equal(o["nov"], one["nov"]) and np.array_equal(o["F"], one["F"])
        np.testing.assert_allclose(o["theta"], one["theta"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(o["ring"], one["ring"], rtol=0, atol=1e-4)
