"""Co-GA safe mutations (SM-G-SUM) on the GPU: the scale kernel against the oracle's fp64 backpropagation, the zero
rule and the floor, determinism and independence of E, K3 with scale rows bit for bit against the oracle's formula,
the wrappers' refusals, and the GA engine: off against the default, on against the oracle, determinism, resume, the
other GA options, and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_novelty as en, ga_safe_mutation as gsm, layout as olayout, philox

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 4343
TINY = 1e-30                     # a floor below every s: c = 1 / s, so s can be read back from the scale
#: parents whose smallest |ReLU input| (over 32 probes x 768 units) is below this are not compared: there a float32
#: forward may take the other side of a ReLU than the fp64 oracle.  On fc_init rows that minimum is typically 1e-5 to
#: 1e-4, so 1e-4 would exclude most parents; 1e-5 is still about 100x the float32 rounding of those O(1) inputs.
MARGIN = 1e-5


def _probe_obs(role, seed=SEED):
    from coevonet_b200 import ops
    states = ops.init_states(seed, en.PROBE_TAG, en.PROBES, "cuda")
    return ops.novelty_probe_obs(states, role)


def _parents(role, seed=SEED):
    """fp32 [7, pitch] on the GPU: two fc_init rows, two sigma-0.05 mutants, and rows with LN gamma x40 / x0.02 and
    fc2 x250 / x0.01."""
    from coevonet_b200 import layout, ops
    in_dim = layout.OBS_DIM[role]
    base = ops.fc_init(in_dim, seed, role, 0, 2, "cuda")
    mut = ops.ga_repopulate(base, layout.fc_dim(in_dim), 0.05, seed, role, 1, 1, 2)
    segs = {name: (off, int(np.prod(shape))) for name, off, shape, _ in olayout.fc_segments(in_dim)[0]}
    scaled = base[0:1].repeat(4, 1)
    for i, (name, f) in enumerate((("ln1.weight", 40.0), ("ln1.weight", 0.02), ("fc2.weight", 250.0),
                                   ("fc2.weight", 0.01))):
        off, n = segs[name]
        scaled[i, off:off + n] *= f
    return torch.cat([base, mut, scaled[:3]]).contiguous(), scaled[3:].contiguous()


def _check_s(c, rows, in_dim, obs):
    """(qualifying parents, largest error over tolerance) of the kernel's s = 1 / c against the oracle."""
    D = olayout.fc_dim(in_dim)
    n_ok, worst = 0, 0.0
    for e in range(rows.shape[0]):
        s_ref, mag, margin = gsm.sensitivity(rows[e, :D], in_dim, obs)
        if margin <= MARGIN:
            continue
        n_ok += 1
        ce = c[e, :D].astype(np.float64)
        s_gpu = np.where(ce == 1.0, np.where(s_ref < 0.5, 0.0, 1.0), 1.0 / ce)
        tol = 1e-4 * s_ref + 1e-5 * mag
        err = np.abs(s_gpu - s_ref)
        worst = max(worst, float((err / np.maximum(tol, 1e-300)).max()))
        bad = np.flatnonzero(err > tol)
        assert bad.size == 0, (e, bad[:5], s_gpu[bad[:5]], s_ref[bad[:5]], mag[bad[:5]])
    return n_ok, worst


@pytest.mark.parametrize("role", ["adversary_0", "agent_0"])
@pytest.mark.parametrize("E", [1, 2, 7])
def test_scale_kernel_against_the_oracle(role, E):
    from coevonet_b200 import layout, ops
    in_dim = layout.OBS_DIM[role]
    obs = _probe_obs(role)
    rows, extra = _parents(role)
    rows = torch.cat([rows, extra])[:E].contiguous() if E < 7 else rows
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    c = ops.ga_safe_scale(rows, in_dim, obs, TINY, status=status)
    assert c.shape == rows.shape and int(status.item()) == 0
    c = c.cpu().numpy()
    assert not c[:, layout.fc_dim(in_dim):].any()
    n_ok, _ = _check_s(c, rows.cpu().numpy(), in_dim, obs.cpu().numpy())
    if E == 7:
        assert n_ok >= 4                                                 # most sampled parents are compared


def test_scaled_extremes_against_the_oracle():
    from coevonet_b200 import layout, ops
    for role in ("adversary_0", "agent_1"):
        in_dim = layout.OBS_DIM[role]
        obs = _probe_obs(role)
        _, extra = _parents(role)
        c = ops.ga_safe_scale(extra, in_dim, obs, TINY).cpu().numpy()
        _check_s(c, extra.cpu().numpy(), in_dim, obs.cpu().numpy())


def test_zero_rule_and_floor():
    from coevonet_b200 import layout, ops
    role, in_dim = "agent_0", 10
    obs = _probe_obs(role)
    rows, _ = _parents(role)
    row = rows[0:1].clone()
    segs = {name: off for name, off, _, _ in olayout.fc_segments(in_dim)[0]}
    u = 41
    row[0, segs["ln2.weight"] + u] = 0.0
    row[0, segs["ln2.bias"] + u] = -1.0                                  # unit u is off on every probe
    c = ops.ga_safe_scale(row, in_dim, obs, 0.01).cpu().numpy()[0]
    assert c[segs["ln2.weight"] + u] == 1.0 and c[segs["ln2.bias"] + u] == 1.0
    assert all(c[segs["output.weight"] + k * 256 + u] == 1.0 for k in range(5))
    assert c[segs["output.bias"]] == np.float32(1.0 / 32.0)
    # the floor: entries whose s is clearly below it get exactly fl32(1 / floor), the others 1 / s
    floor = 0.5
    c = ops.ga_safe_scale(rows[:2], in_dim, obs, floor).cpu().numpy()
    at = np.float32(1) / np.float32(floor)
    D = layout.fc_dim(in_dim)
    for e in range(2):
        s_ref, mag, _ = gsm.sensitivity(rows[e].cpu().numpy()[:D], in_dim, obs.cpu().numpy())
        low = (s_ref > 1e-3 * floor) & (s_ref + 1e-4 * s_ref + 1e-5 * mag < floor)
        high = s_ref - 1e-4 * s_ref - 1e-5 * mag > floor
        assert low.sum() > 100 and high.sum() > 100
        assert np.all(c[e, :D][low] == at)
        assert np.all(c[e, :D][high] < at)
        assert np.all(c[e, :D] <= at)


def test_deterministic_and_independent_of_E():
    from coevonet_b200 import ops
    for role in ("adversary_0", "agent_0"):
        in_dim = 8 if role == "adversary_0" else 10
        obs = _probe_obs(role)
        rows, _ = _parents(role)
        c7 = ops.ga_safe_scale(rows, in_dim, obs, 0.01)
        assert torch.equal(c7.view(torch.int32), ops.ga_safe_scale(rows, in_dim, obs, 0.01).view(torch.int32))
        for e in range(7):
            c1 = ops.ga_safe_scale(rows[e:e + 1], in_dim, obs, 0.01)
            assert torch.equal(c1[0].view(torch.int32), c7[e].view(torch.int32)), (role, e)


def test_nonfinite_sets_the_status():
    from coevonet_b200 import ops
    obs = _probe_obs("agent_0")
    rows, _ = _parents("agent_0")
    bad = rows[:2].clone()
    bad[1, 5000] = float("nan")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.ga_safe_scale(bad, 10, obs, 0.01, status=status)
    assert int(status.item()) != 0
    status.zero_()
    ops.ga_safe_scale(rows[:2], 10, obs, 0.01, status=status)
    assert int(status.item()) == 0


# ---------------------------------------------------------------------------------------------------------------
# K3 with scale rows
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rate,row0", [(0.0, 0), (0.0, 5), (0.6, 0), (0.6, 13)])
def test_k3_safe_against_the_oracle(rate, row0):
    from coevonet_b200 import layout, ops
    role, in_dim = "agent_1", 10
    D = layout.fc_dim(in_dim)
    rows, _ = _parents(role)
    elites = rows[:3].contiguous()
    scale = ops.ga_safe_scale(elites, in_dim, _probe_obs(role), 0.01)
    n = 40
    noise = torch.empty((n, elites.shape[1]), dtype=torch.float32, device="cuda")
    got = ops.ga_repopulate(elites, D, 0.05, SEED, role, 3, row0, n, noise_out=noise, crossover_rate=rate,
                            scale=scale).cpu().numpy()
    members = np.arange(row0, row0 + n)
    want = gsm.children(elites.cpu().numpy()[:, :D], scale.cpu().numpy(), 0.05, noise.cpu().numpy()[:, :D], members,
                        rate, SEED, layout.ROLE_ID[role], 3)
    assert np.array_equal(got[:, :D].view(np.uint32), want.view(np.uint32))
    assert not got[:, D:].any()
    if row0 == 0:
        assert np.array_equal(got[0], elites[0].cpu().numpy())          # row 0: the best, unmutated
    # a scale row of ones is the plain K3 bit for bit
    ones = torch.ones_like(elites)
    plain = ops.ga_repopulate(elites, D, 0.05, SEED, role, 3, row0, n, crossover_rate=rate)
    assert torch.equal(ops.ga_repopulate(elites, D, 0.05, SEED, role, 3, row0, n, crossover_rate=rate,
                                         scale=ones).view(torch.int32), plain.view(torch.int32))


def test_k3_safe_with_device_sigma():
    from coevonet_b200 import layout, ops
    rows, _ = _parents("adversary_0")
    elites = rows[:2].contiguous()
    D = layout.fc_dim(8)
    scale = ops.ga_safe_scale(elites, 8, _probe_obs("adversary_0"), 0.01)
    sig = torch.tensor([0.07], dtype=torch.float64, device="cuda")
    assert torch.equal(ops.ga_repopulate(elites, D, sig, 9, "adversary_0", 2, 0, 9, scale=scale),
                       ops.ga_repopulate(elites, D, 0.07, 9, "adversary_0", 2, 0, 9, scale=scale))


def test_wrappers_refuse_bad_arguments():
    from coevonet_b200 import _lib, layout, ops
    rows, _ = _parents("agent_0")
    obs = _probe_obs("agent_0")
    D = layout.fc_dim(10)
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows.cpu(), 10, obs, 0.01)
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows, 10, obs.cpu(), 0.01)
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows, 8, obs, 0.01)                           # probes of the other in_dim
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows, 9, obs, 0.01)
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows[:, :D - 1], 10, obs, 0.01)
    for floor in (0.0, -1.0, float("nan"), float("inf")):
        with pytest.raises(_lib.CevError):
            ops.ga_safe_scale(rows, 10, obs, floor)
    with pytest.raises(_lib.CevError):
        ops.ga_safe_scale(rows, 10, obs, 0.01, out=torch.empty((6, rows.shape[1]), device="cuda"))
    scale = ops.ga_safe_scale(rows, 10, obs, 0.01)
    with pytest.raises(_lib.CevError):
        ops.ga_repopulate(rows, D, 0.05, 1, "agent_0", 0, 0, 4, scale=scale[:3].contiguous())
    with pytest.raises(_lib.CevError):
        ops.ga_repopulate(rows, D, 0.05, 1, "agent_0", 0, 0, 4, scale=scale.cpu())
    with pytest.raises(_lib.CevError):
        ops.ga_repopulate(rows, D, 0.05, 1, "agent_0", 0, 0, 4, scale=scale.double())
    assert ops.ga_safe_scale(rows[:0], 10, obs, 0.01).shape == (0, rows.shape[1])


# ---------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------
def _args(P, E=2, **opts):
    a = types.SimpleNamespace(
        algorithm="GA", generations=8, population=P, hof_size=3, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=4,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=E, reference_compat=True, init_states="device", seed=SEED, plots=False,
        record_history=False)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _rows(P, hof, dev="cuda", row0=0, n=None):
    from coevonet_b200 import layout, ops
    n = P if n is None else n
    pop, hof_rows, founder = {}, {}, {}
    for r in ROLES:
        in_dim = layout.OBS_DIM[r]
        pop[r] = ops.fc_init(in_dim, 5, r, row0, n, dev).cpu()
        hof_rows[r] = ops.fc_init(in_dim, 6, r, 0, hof, dev).cpu()
        founder[r] = ops.fc_init(in_dim, 7, r, 0, 1, dev)[0].cpu()
    return pop, hof_rows, founder


def _engine(P, **opts):
    from coevonet_b200 import engine
    args = _args(P, **opts)
    pop, hof, founder = _rows(P, int(args.hof_size))
    return engine.GAEngine(args, torch.device("cuda", 0), pop, hof, founder)


SAFE = dict(ga_safe_mutation=True, ga_safe_mutation_floor=0.02)


def _bits(eng):
    eng.check_status()
    out = {"gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["pop_" + r] = eng.pop[r].cpu().numpy().view(np.uint32)
        out["hof_" + r] = eng.hof[r].cpu().numpy().view(np.uint32)
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["elite_" + r] = eng.elite_ids[r].cpu().numpy()
        if eng.safe:
            out["scale_" + r] = eng.safe_scale[r].cpu().numpy().view(np.uint32)
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_off_equals_the_default_engine():
    plain = _engine(64)
    off = _engine(64, ga_safe_mutation=False)
    for _ in range(3):
        plain.step(sync=False)
        off.step(sync=False)
        _same(_bits(plain), _bits(off))
    assert off.novelty_probe_obs is None


def _follows_the_oracle(eng, P, gens, rate=0.0):
    from coevonet_b200 import layout, ops
    obs = {r: _probe_obs(r) for r in ROLES}
    for r in ROLES:
        assert torch.equal(eng.novelty_probe_obs[r], obs[r])
    for g in range(gens):
        before = {r: eng.pop[r].clone() for r in ROLES}
        eng.step()
        h = eng.history[g]
        sig = h["sigma"]                                                 # the mutation power of generation g
        for r in ROLES:
            in_dim = layout.OBS_DIM[r]
            D = layout.fc_dim(in_dim)
            elites = before[r][torch.from_numpy(h["elite_ids"][r]).cuda()].contiguous()
            scale = ops.ga_safe_scale(elites, in_dim, obs[r], SAFE["ga_safe_mutation_floor"])
            assert torch.equal(eng.safe_scale[r], scale), (g, r)
            members = np.arange(P)
            z = philox.normals(SEED, philox.KIND_GA, layout.ROLE_ID[r], g, members, D)
            noise = torch.empty((P, elites.shape[1]), dtype=torch.float32, device="cuda")
            ops.ga_repopulate(elites, D, sig[r], SEED, r, g, 0, P, noise_out=noise, crossover_rate=rate, scale=scale)
            np.testing.assert_allclose(noise.cpu().numpy()[1:, :D], z[1:], rtol=0, atol=3e-6)
            want = gsm.children(elites.cpu().numpy()[:, :D], scale.cpu().numpy(), sig[r], noise.cpu().numpy()[:, :D],
                                members, rate, SEED, layout.ROLE_ID[r], g)
            assert np.array_equal(eng.pop[r].cpu().numpy()[:, :D].view(np.uint32), want.view(np.uint32)), (g, r)
            c = scale.cpu().numpy()[:, :D]
            st = h["safe_mutation_scale"][r]
            assert st["min"] == float(c.min()) and st["max"] == float(c.max())
            assert st["n_floor"] == int((c == np.float32(1) / np.float32(SAFE["ga_safe_mutation_floor"])).sum())
            assert 0 < st["min"] <= st["mean"] <= st["max"] <= 1 / SAFE["ga_safe_mutation_floor"] * (1 + 1e-6)


def test_generations_match_the_oracle():
    """Every child of 3 generations is the oracle's formula on the engine's elites, their ga_safe_scale rows and the
    kernel's normals."""
    P = 48
    _follows_the_oracle(_engine(P, record_history=True, **SAFE), P, 3)


def test_deterministic_and_resume_is_bit_identical():
    a, b = _engine(64, **SAFE), _engine(64, **SAFE)
    for _ in range(2):
        a.step(sync=False)
        b.step(sync=False)
    _same(_bits(a), _bits(b))
    sd = a.state_dict()
    for _ in range(2):
        a.step(sync=False)
    c = _engine(64, **SAFE)
    c.load_state_dict(sd)
    for _ in range(2):
        c.step(sync=False)
    _same(_bits(a), _bits(c))


@pytest.mark.parametrize("opts", [dict(ga_novelty_weight=0.5, ga_novelty_k=4, ga_novelty_archive=5),
                                  dict(crossover_rate=0.3), dict(adaptive=True), dict(fitness_sharing=False),
                                  dict(reference_compat=False, fitness_sharing=True),
                                  dict(play_discarded_hof_games=True)],
                         ids=["novelty", "crossover", "adaptive", "no_sharing", "no_reference_compat",
                              "discarded_hof_games"])
def test_composes_with_the_other_options(opts):
    P = 40
    eng = _engine(P, record_history=True, **dict(SAFE, **opts))
    _follows_the_oracle(eng, P, 2, opts.get("crossover_rate", 0.0))
    eng.check_status()


# ---------------------------------------------------------------------------------------------------------------
# two GPUs
# ---------------------------------------------------------------------------------------------------------------
def _worker(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from coevonet_b200 import engine
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    comm = engine.Comm()
    shard = engine.Shard(P, comm.rank, comm.world)
    args = _args(P, record_history=True, **SAFE)
    pop, hof, founder = _rows(P, int(args.hof_size), dev, shard.row0, shard.n_local)
    eng = engine.GAEngine(args, dev, pop, hof, founder, comm=comm)
    for _ in range(3):
        eng.step()
    q.put((rank, dict(row0=shard.row0, n_local=shard.n_local,
                      elite_ids=np.stack([eng.history[g]["elite_ids"][r] for g in range(3) for r in ROLES]),
                      fitness=np.stack([eng.history[g]["fitness"][r] for g in range(3) for r in ROLES]),
                      scale=np.concatenate([eng.safe_scale[r].cpu().numpy() for r in ROLES], axis=1),
                      hof=np.concatenate([eng.hof[r].cpu().numpy() for r in ROLES], axis=1),
                      pop=np.concatenate([eng.pop[r].cpu().numpy() for r in ROLES], axis=1))))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _launch(world, P, port):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, P, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    outs = dict(q.get(timeout=600) for _ in range(world))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return [outs[r] for r in range(world)]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_safe_mutation_sharded_over_two_gpus_equal_one_gpu():
    P = 387                                        # 194 + 193 rows
    one = _launch(1, P, 29761)[0]
    two = _launch(2, P, 29762)
    for o in two:
        for key in ("elite_ids", "scale", "hof"):
            assert np.array_equal(o[key], one[key]), key
        np.testing.assert_allclose(o["fitness"], one["fitness"], rtol=1e-12, atol=0)
        assert np.array_equal(o["pop"], one["pop"][o["row0"]:o["row0"] + o["n_local"]])
