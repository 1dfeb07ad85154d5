"""The opt-in Co-ES update kernels through the C ABI (mirrored K5 / K6, centered ranks, fused apply) against the
oracle, and the ES engine with the options on: determinism, resume, defaults unchanged, two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_options as oes, layout as olayout, philox, weights

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 1870300
ALL_ON = dict(mirrored_sampling=True, fitness_shaping="centered_rank", es_optimizer="adam", learning_rate=0.01,
              l2_coeff=0.005)


def _theta(in_dim, seed=43):
    from coevonet_b200 import layout
    row = np.zeros(layout.fc_pitch(in_dim), dtype=np.float32)
    row[:layout.fc_dim(in_dim)] = weights.make_fc_rows(1, in_dim, seed, ln_jitter=0.02)[0]
    return row


# ---------------------------------------------------------------------------------------------------------------
# mirrored K5
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("role,in_dim", [("agent_1", 10), ("adversary_0", 8)])
def test_es_perturb_mirrored(role, in_dim):
    from coevonet_b200 import layout, ops
    D, pitch = layout.fc_dim(in_dim), layout.fc_pitch(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    P, gen, sigma = 96, 3, 0.05
    theta = _theta(in_dim)
    dev_theta = torch.from_numpy(theta).cuda()
    noise = torch.full((P, pitch), 7.0, device="cuda")
    rows = ops.es_perturb_mirrored(dev_theta, in_dim, sigma, SEED, role, gen, 0, P, noise_out=noise)
    sz = noise.cpu().numpy()
    # one draw per pair: the odd member carries exactly the negated normals of the even one
    assert np.array_equal(sz[1::2], -sz[0::2])
    z_dev = sz[0::2, :D]
    z = philox.normals(SEED, oes.KIND_ES_MIRROR, philox.ROLE_ID[role], gen, np.arange(P // 2), D)
    np.testing.assert_allclose(z_dev[:, pidx], z[:, pidx], rtol=0, atol=3e-6)
    mask = np.ones(D, bool)
    mask[pidx] = False
    assert np.all(z_dev[:, mask] == 0) and np.all(sz[:, D:] == 0)
    assert abs(z_dev[:, pidx].mean()) < 5e-3 and abs(z_dev[:, pidx].std() - 1) < 5e-3
    # rows bit-exact against the restatement given the device normals
    want, _ = oes.es_perturb_mirrored(theta[:D], sigma, z_dev, pidx, 0, P)
    got = rows.cpu().numpy()
    assert np.array_equal(got[:, :D], want)
    assert np.all(got[:, D:] == 0)
    # the default ES stream is untouched: plain K5 is another draw
    plain = ops.es_perturb(dev_theta, in_dim, sigma, SEED, role, gen, 0, 2)
    assert not torch.equal(plain, rows[:2])
    # shard edges: a block starting / ending inside a pair writes only its own rows
    for row0, n in ((1, 10), (5, 1), (2, 7), (0, 1), (95, 1), (33, 63)):
        part_noise = torch.zeros((n, pitch), device="cuda")
        part = ops.es_perturb_mirrored(dev_theta, in_dim, sigma, SEED, role, gen, row0, n, noise_out=part_noise)
        assert torch.equal(part, rows[row0:row0 + n]), (row0, n)
        assert torch.equal(part_noise, noise[row0:row0 + n]), (row0, n)
    # nothing outside the block is written
    out = torch.full((P + 2, pitch), 3.0, device="cuda")
    ops.es_perturb_mirrored(dev_theta, in_dim, sigma, SEED, role, gen, 3, 5, out=out[1:6])
    assert torch.equal(out[1:6], rows[3:8])
    assert bool((out[0] == 3.0).all()) and bool((out[6:] == 3.0).all())


# ---------------------------------------------------------------------------------------------------------------
# mirrored K6, noise regenerated
# ---------------------------------------------------------------------------------------------------------------
def _fma32(a, b, c):
    """Correctly rounded float32 fmaf(a, b, c), elementwise: the fp64 product is exact, the fp64 sum carries its
    exact error (TwoSum), and a sum that lands on a float32 midpoint is rounded toward the error."""
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    bb = s - p
    e = (p - (s - bb)) + (c64 - bb)
    r = s.astype(np.float32)
    up, dn = np.nextafter(r, np.float32(np.inf)), np.nextafter(r, np.float32(-np.inf))
    r = np.where((s == (r.astype(np.float64) + up) / 2) & (e > 0), up, r)
    r = np.where((s == (r.astype(np.float64) + dn) / 2) & (e < 0), dn, r)
    return r


def _es_update_mirrored_oracle(fitness, z_pairs, sigma, lr, n_total, row0):
    """K6 mirrored in the kernel's order: per MEMBER, fmaf(s_i * fl(sigma z_q), F_i, acc) in row order within the
    splits (even global starts, cev_es_update_mirrored_f32), then the splits summed in order, times the fp32
    coefficient lr / (n_total sigma)."""
    n = len(fitness)
    n_split = min(16, max(1, (n + 63) // 64))
    base = row0 & ~1
    span = row0 + n - base
    per = (-(-span // n_split) + 1) & ~1
    sig = np.float32(sigma)
    total = np.zeros(z_pairs.shape[1], np.float32)
    for sp in range(n_split):
        acc = np.zeros(z_pairs.shape[1], np.float32)
        for r in range(max(base + sp * per, row0) - row0, min(base + (sp + 1) * per, row0 + n) - row0):
            c = row0 + r
            a = (sig * z_pairs[c >> 1]).astype(np.float32)
            acc = _fma32(a if c % 2 == 0 else -a, np.full_like(a, np.float32(fitness[r])), acc)
        total = (total + acc).astype(np.float32)
    coef = np.float32(float(np.float32(lr)) / (n_total * float(sig)))        # the C ABI takes lr as fp32
    return (coef * total).astype(np.float32)


def test_fma32_emulation():
    rng = np.random.default_rng(0)
    a = rng.normal(size=100000).astype(np.float32)
    b = rng.normal(size=100000).astype(np.float32)
    c = rng.normal(size=100000).astype(np.float32)
    from fractions import Fraction

    def round32(x):                       # exact value -> nearest float32, ties to even
        r = np.float32(float(x))
        cands = (np.nextafter(r, np.float32(-np.inf)), r, np.nextafter(r, np.float32(np.inf)))
        return min(cands, key=lambda y: (abs(Fraction(float(y)) - x), int(np.array(y).view(np.uint32)) & 1))

    got = _fma32(a, b, c)
    for i in range(0, 100000, 997):
        assert got[i] == round32(Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i])))
    # (1 + 2^-23) + 2^-24 (1 - 2^-23)(1 + 2^-23): exactly 2^-70 below a float32 midpoint, which is where the fp64
    # sum lands; a second rounding of it (ties to even) would go up, the fma stays down
    c1 = np.array([np.float32(1 + 2.0 ** -23)])
    x = _fma32(np.array([np.float32(2.0 ** -24 * (1 - 2.0 ** -23))]), np.array([np.float32(1 + 2.0 ** -23)]), c1)
    assert (c1.astype(np.float64) + 2.0 ** -24 * (1 - 2.0 ** -46)).astype(np.float32)[0] != c1[0]
    assert x[0] == c1[0]


@pytest.mark.parametrize("row0,n_rows", [(0, 300), (75, 150), (0, 64), (3, 1)])
def test_es_update_mirrored_bit_identical_to_the_per_member_order(row0, n_rows):
    from coevonet_b200 import layout, ops
    in_dim, role, gen, sigma, lr, P = 10, "agent_0", 5, 0.05, 0.1, 300
    D = layout.fc_dim(in_dim)
    pitch = layout.fc_pitch(in_dim)
    theta = torch.from_numpy(_theta(in_dim, 7)).cuda()
    noise = torch.zeros((P, pitch), device="cuda")
    ops.es_perturb_mirrored(theta, in_dim, sigma, SEED, role, gen, 0, P, noise_out=noise)
    z_pairs = noise.cpu().numpy()[0::2]
    fit = np.random.default_rng(row0).normal(-20, 5, n_rows)
    got = ops.es_update_mirrored(torch.from_numpy(fit).cuda(), in_dim, sigma, lr, P, SEED, role, gen, row0)
    want = _es_update_mirrored_oracle(fit, z_pairs, sigma, lr, P, row0)
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32))
    assert np.all(got.cpu().numpy()[D:] == 0)


def test_es_update_mirrored_agrees_with_the_members_form():
    """Same tolerance as test_es_update_from_members_matches_regenerated_update: the members form reads
    sigma*z back as member - theta, one rounding of the perturbation's add per term."""
    from coevonet_b200 import layout, ops
    P, in_dim, sigma, lr, seed = 300, 10, 0.05, 0.1, 77
    theta = torch.from_numpy(_theta(in_dim, 5)).cuda()
    members = ops.es_perturb_mirrored(theta, in_dim, sigma, seed, "agent_1", 3, 0, P)
    fit = torch.randn(P, dtype=torch.float64, device="cuda")
    want = ops.es_update_mirrored(fit, in_dim, sigma, lr, P, seed, "agent_1", 3, 0)
    got = ops.es_update_members(fit, members, theta, in_dim, sigma, lr, P)
    scale = float(want.abs().max())
    assert scale > 0
    assert float((got - want).abs().max()) <= 1e-6 * scale + 1e-9
    assert torch.equal(got == 0, want == 0)
    # sharded partial sums with a pair cut by the boundary add up to the whole
    d0 = ops.es_update_mirrored(fit[:151].contiguous(), in_dim, sigma, lr, P, seed, "agent_1", 3, 0)
    d1 = ops.es_update_mirrored(fit[151:].contiguous(), in_dim, sigma, lr, P, seed, "agent_1", 3, 151)
    assert float((d0 + d1 - want).abs().max()) <= 1e-6 * scale


# ---------------------------------------------------------------------------------------------------------------
# centered ranks
# ---------------------------------------------------------------------------------------------------------------
def test_centered_ranks_bit_exact():
    from coevonet_b200 import ops
    rng = np.random.default_rng(11)
    cases = [np.array([2.5]), np.array([1.0, 1.0]), np.array([np.nan, -0.0, 0.0, -np.inf, np.inf, 3.0, np.nan])]
    for P in (7, 1000, 2049, 65536):
        f = np.round(rng.normal(-30, 4, P), 1)                      # many ties
        f[rng.random(P) < 0.01] = np.nan
        f[rng.random(P) < 0.01] = 0.0
        f[rng.random(P) < 0.01] = -0.0
        cases.append(f)
    cases.append(rng.normal(size=8192))
    for f in cases:
        want = oes.centered_ranks(f)
        got = ops.centered_ranks(torch.from_numpy(f).cuda()).cpu().numpy()
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), len(f)
    f = cases[-2]
    dev = torch.from_numpy(f).cuda()
    want = oes.centered_ranks(f)
    for row0, n in ((32768, 32768), (12345, 777), (65535, 1), (0, 0)):
        got = ops.centered_ranks(dev, row0, n).cpu().numpy()
        assert np.array_equal(got, want[row0:row0 + n]), (row0, n)


# ---------------------------------------------------------------------------------------------------------------
# fused apply
# ---------------------------------------------------------------------------------------------------------------
def test_es_apply_bit_exact():
    from coevonet_b200 import layout, ops
    in_dims = [10, 10, 8]
    mask = np.concatenate([np.isin(np.arange(layout.fc_pitch(d)), olayout.fc_perturbable_index(d)) for d in in_dims])
    n = mask.size
    rng = np.random.default_rng(3)
    theta = rng.normal(0, 0.2, n).astype(np.float32)
    m = np.where(mask, 0, -5).astype(np.float32)
    v = np.where(mask, 0, 9).astype(np.float32)
    dt, dm, dv = (torch.from_numpy(x.copy()).cuda() for x in (theta, m, v))
    for t in range(1, 7):
        g = rng.normal(0, 0.1, n).astype(np.float32)
        g[rng.random(n) < 0.01] = 0.0
        ops.es_apply(dt, torch.from_numpy(g).cuda(), in_dims, optimizer="adam", lr=0.01, l2_coeff=0.005, t=t,
                     m=dm, v=dv)
        theta, m, v = oes.es_apply(theta, g, mask, "adam", 0.01, 0.005, t, m, v)
        for got, want in ((dt, theta), (dm, m), (dv, v)):
            assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32)), t
    g = rng.normal(0, 0.1, n).astype(np.float32)
    ops.es_apply(dt, torch.from_numpy(g).cuda(), in_dims, optimizer="sgd", lr=0.1, l2_coeff=0.02)
    theta, _, _ = oes.es_apply(theta, g, mask, "sgd", 0.1, 0.02)
    assert np.array_equal(dt.cpu().numpy().view(np.uint32), theta.view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------
def _args(P, E=4, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=4, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=True, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=E, reference_compat=True, init_states="device", seed=31337, plots=False,
        record_history=False)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _engine(P, **opts):
    from coevonet_b200 import engine, layout, ops
    theta = {r: ops.fc_init(layout.OBS_DIM[r], 5, r, 0, 1, "cuda")[0].cpu() for r in ROLES}
    return engine.ESEngine(_args(P, **opts), torch.device("cuda", 0), theta)


def _bits(eng):
    eng.check_status()
    out = {"theta": eng.theta_cat.cpu().numpy().view(np.uint32), "gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["rew_" + r] = eng.rewards[r].cpu().numpy()
    if eng.adam_m is not None:
        out["m"] = eng.adam_m.cpu().numpy().view(np.uint32)
        out["v"] = eng.adam_v.cpu().numpy().view(np.uint32)
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("regenerate", [False, True])
def test_engine_all_options_deterministic(regenerate):
    runs = []
    for _ in range(2):
        eng = _engine(64, update_from_members=not regenerate, **ALL_ON)
        for _ in range(3):
            eng.step(sync=False)
        runs.append(_bits(eng))
        assert eng.shaped_fitness["agent_0"].shape == (64,)
    _same(*runs)
    assert np.any(runs[0]["m"] != 0)


def test_engine_all_options_resume_bit_exact(tmp_path):
    full = _engine(64, **ALL_ON)
    for _ in range(4):
        full.step(sync=False)
    first = _engine(64, **ALL_ON)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "es.pt")
    second = _engine(64, **ALL_ON)
    second.load_state_dict(torch.load(tmp_path / "es.pt", weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    _same(_bits(full), _bits(second))


def test_engine_defaults_equal_an_engine_without_the_options():
    plain = _engine(64)
    explicit = _engine(64, mirrored_sampling=False, fitness_shaping="none", es_optimizer="sgd", l2_coeff=0.0)
    for _ in range(3):
        plain.step(sync=False)
        explicit.step(sync=False)
    _same(_bits(plain), _bits(explicit))


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
    eng = engine.ESEngine(_args(P, E, **ALL_ON), dev, theta, comm=comm)
    eng.evaluate()
    eng.update()
    out = dict(rewards=np.stack([comm.all_gather_rows(eng.rewards[r], eng.shard).cpu().numpy() for r in ROLES]),
               shaped=np.stack([comm.all_gather_rows(eng.shaped_fitness[r], eng.shard).cpu().numpy() for r in ROLES]),
               delta=eng.delta_cat.cpu().numpy(), theta=eng.theta_cat.cpu().numpy())
    if rank == 0:
        q.put(out)
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
    out = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    return out


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_es_options_sharded_over_two_gpus_equal_one_gpu():
    P, E = 386, 16                                 # 193 + 193 rows: the pair (192, 193) is cut by the boundary
    one = _launch(1, P, E, 29711)
    two = _launch(2, P, E, 29712)
    assert np.array_equal(one["rewards"], two["rewards"])
    assert np.array_equal(one["shaped"], two["shaped"])
    scale = np.abs(one["delta"]).max()
    assert np.abs(one["delta"] - two["delta"]).max() <= 1e-5 * scale    # all-reduce summation order only
