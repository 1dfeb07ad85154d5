"""Separable NES through the C ABI (diag K5 / K6 / apply) against the isotropic kernels and the oracle, and the ES
engine with ``es_distribution="separable"``: determinism, resume, defaults unchanged, two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import layout as olayout, snes, weights

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_gpu_es_options import _fma32  # noqa: E402

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 1870300
SNES_ALL = dict(es_distribution="separable", mirrored_sampling=True, fitness_shaping="centered_rank",
                learning_rate=1.0)


def _theta(in_dim, seed=43):
    from coevonet_b200 import layout
    row = np.zeros(layout.fc_pitch(in_dim), dtype=np.float32)
    row[:layout.fc_dim(in_dim)] = weights.make_fc_rows(1, in_dim, seed, ln_jitter=0.02)[0]
    return row


def _pert(in_dim):
    from coevonet_b200 import layout
    m = np.zeros(layout.fc_pitch(in_dim), bool)
    m[olayout.fc_perturbable_index(in_dim)] = True
    return m


def _sigma_row(in_dim, value):
    return np.where(_pert(in_dim), np.float32(value), np.float32(0)).astype(np.float32)


# ---------------------------------------------------------------------------------------------------------------
# diag K5
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mirrored", [False, True])
@pytest.mark.parametrize("role,in_dim", [("agent_1", 10), ("adversary_0", 8)])
def test_perturb_diag_with_sigma0_is_the_isotropic_k5(role, in_dim, mirrored):
    from coevonet_b200 import layout, ops
    pitch = layout.fc_pitch(in_dim)
    gen, sigma0 = 3, 0.05
    theta = torch.from_numpy(_theta(in_dim)).cuda()
    sigma = torch.from_numpy(_sigma_row(in_dim, sigma0)).cuda()
    iso = ops.es_perturb_mirrored if mirrored else ops.es_perturb
    for row0, n in ((0, 96), (3, 17), (1, 1), (33, 64)):
        n_iso, n_diag = torch.full((n, pitch), 7.0, device="cuda"), torch.full((n, pitch), 9.0, device="cuda")
        want = iso(theta, in_dim, sigma0, SEED, role, gen, row0, n, noise_out=n_iso)
        got = ops.es_perturb_diag(theta, sigma, in_dim, SEED, role, gen, row0, n, mirrored=mirrored, noise_out=n_diag)
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), (row0, n)
        assert torch.equal(n_diag, n_iso), (row0, n)


@pytest.mark.parametrize("mirrored", [False, True])
def test_perturb_diag_with_a_random_sigma_matches_the_oracle(mirrored):
    from coevonet_b200 import layout, ops
    in_dim, role, gen, P, row0 = 10, "agent_0", 2, 40, 5
    D, pitch = layout.fc_dim(in_dim), layout.fc_pitch(in_dim)
    pidx = olayout.fc_perturbable_index(in_dim)
    theta = _theta(in_dim, 9)
    rng = np.random.default_rng(4)
    sigma = np.where(_pert(in_dim), rng.uniform(0.001, 0.2, pitch), 0).astype(np.float32)
    noise = torch.zeros((P, pitch), device="cuda")
    got = ops.es_perturb_diag(torch.from_numpy(theta).cuda(), torch.from_numpy(sigma).cuda(), in_dim, SEED, role, gen,
                              row0, P, mirrored=mirrored, noise_out=noise).cpu().numpy()
    sz = noise.cpu().numpy()
    if mirrored:                                  # rows 0, 1 of the block are members 5 (odd) and 6 (even)
        assert np.array_equal(sz[2::2], -sz[1:-1:2]) and not np.array_equal(sz[0], -sz[1])
    want, _ = snes.perturb(theta[:D], sigma[:D], sz[:, :D], pidx)      # noise_out holds s z
    assert np.array_equal(got[:, :D].view(np.uint32), want.view(np.uint32))
    assert np.all(got[:, D:] == 0)


# ---------------------------------------------------------------------------------------------------------------
# diag K6
# ---------------------------------------------------------------------------------------------------------------
def _splits(row0, n, mirrored):
    n_split = min(16, max(1, (n + 63) // 64))
    if not mirrored:
        per = -(-n // n_split)
        return [(sp * per, min(n, sp * per + per)) for sp in range(n_split)]
    base = row0 & ~1
    per = (-(-(row0 + n - base) // n_split) + 1) & ~1
    return [(max(base + sp * per, row0) - row0, min(base + (sp + 1) * per, row0 + n) - row0) for sp in range(n_split)]


def _update_diag_oracle(fitness, sz, n_total, row0, mirrored):
    """diag K6 in the kernel's order: per member, fmaf(s z, F, acc) and fmaf(fl(fl(z z) - 1), F, acc2) in row order
    within the documented splits, the splits summed in order, times fl32(1 / n_total).  ``sz``: the members' s z."""
    one = np.float32(1)
    tot_mu = np.zeros(sz.shape[1], np.float32)
    tot_sg = np.zeros(sz.shape[1], np.float32)
    for lo, hi in _splits(row0, len(fitness), mirrored):
        a_mu = np.zeros(sz.shape[1], np.float32)
        a_sg = np.zeros(sz.shape[1], np.float32)
        for r in range(lo, hi):
            z = sz[row0 + r]
            f = np.full_like(z, np.float32(fitness[r]))
            a_mu = _fma32(z, f, a_mu)
            a_sg = _fma32((z * z - one).astype(np.float32), f, a_sg)
        tot_mu = (tot_mu + a_mu).astype(np.float32)
        tot_sg = (tot_sg + a_sg).astype(np.float32)
    inv_n = np.float32(1.0 / n_total)
    pert = _pert(10)[:sz.shape[1]]            # the kernel writes zeros off the Linear entries (there z^2 - 1 = -1)
    return (np.where(pert, inv_n * tot_mu, 0).astype(np.float32),
            np.where(pert, inv_n * tot_sg, 0).astype(np.float32))


@pytest.mark.parametrize("mirrored", [False, True])
@pytest.mark.parametrize("row0,n_rows", [(0, 300), (75, 150), (0, 64), (3, 1)])
def test_update_diag_bit_identical_to_the_per_member_order(row0, n_rows, mirrored):
    from coevonet_b200 import layout, ops
    in_dim, role, gen, P = 10, "agent_0", 5, 300
    D, pitch = layout.fc_dim(in_dim), layout.fc_pitch(in_dim)
    theta = torch.from_numpy(_theta(in_dim, 7)).cuda()
    noise = torch.zeros((P, pitch), device="cuda")
    (ops.es_perturb_mirrored if mirrored else ops.es_perturb)(theta, in_dim, 0.05, SEED, role, gen, 0, P,
                                                              noise_out=noise)
    sz = noise.cpu().numpy()
    fit = np.random.default_rng(row0 + n_rows).normal(-20, 5, n_rows)
    g_mu, g_sigma = ops.es_update_diag(torch.from_numpy(fit).cuda(), in_dim, P, SEED, role, gen, row0,
                                       mirrored=mirrored)
    want_mu, want_sg = _update_diag_oracle(fit, sz, P, row0, mirrored)
    assert np.array_equal(g_mu.cpu().numpy().view(np.uint32), want_mu.view(np.uint32))
    assert np.array_equal(g_sigma.cpu().numpy().view(np.uint32), want_sg.view(np.uint32))
    ln = ~_pert(in_dim)
    assert np.all(g_mu.cpu().numpy()[ln] == 0) and np.all(g_sigma.cpu().numpy()[ln] == 0)
    assert np.all(g_mu.cpu().numpy()[D:] == 0)


@pytest.mark.parametrize("mirrored", [False, True])
def test_update_diag_mu_gradient_is_the_isotropic_delta(mirrored):
    """At sigma = sigma0 the SNES mu step lr * sigma0 * g_mu is K6's delta at the learning rate lr * sigma0:
    (lr sigma0) / (n sigma0) * sum_i (sigma0 z_i) F_i = lr sigma0 / n * sum_i z_i F_i, up to fp32 rounding."""
    from coevonet_b200 import ops
    P, in_dim, sigma0, lr = 300, 8, 0.05, 1.0
    fit = torch.randn(P, dtype=torch.float64, device="cuda") * 5 - 20
    delta = (ops.es_update_mirrored if mirrored else ops.es_update)(fit, in_dim, sigma0, lr * sigma0, P, SEED,
                                                                    "adversary_0", 4, 0)
    g_mu, _ = ops.es_update_diag(fit, in_dim, P, SEED, "adversary_0", 4, 0, mirrored=mirrored)
    got = lr * sigma0 * g_mu.double()
    scale = float(delta.abs().max())
    assert scale > 0
    assert float((got - delta.double()).abs().max()) <= 2e-5 * scale
    assert torch.equal(g_mu == 0, delta == 0)


# ---------------------------------------------------------------------------------------------------------------
# diag apply
# ---------------------------------------------------------------------------------------------------------------
def test_apply_diag_matches_the_oracle():
    from coevonet_b200 import layout, ops
    in_dims = [10, 10, 8]
    etas = [0.05, 0.3, 1.5]
    mask = np.concatenate([_pert(d) for d in in_dims])
    eta = np.concatenate([np.full(layout.fc_pitch(d), e) for d, e in zip(in_dims, etas)])
    n = mask.size
    rng = np.random.default_rng(8)
    theta = rng.normal(0, 0.2, n).astype(np.float32)
    sigma = np.where(mask, rng.uniform(0.01, 0.09, n), rng.normal(0, 1, n)).astype(np.float32)   # junk off mask
    smin, smax = 0.005, 0.1
    dt, ds = torch.from_numpy(theta.copy()).cuda(), torch.from_numpy(sigma.copy()).cuda()
    for step in range(3):
        g_mu = rng.normal(0, 3, n).astype(np.float32)
        g_sg = rng.normal(0, 2, n).astype(np.float32)
        ops.es_apply_diag(dt, ds, torch.from_numpy(g_mu).cuda(), torch.from_numpy(g_sg).cuda(), in_dims, lr=0.7,
                          sigma_lr=etas, sigma_min=smin, sigma_max=smax)
        theta, sigma_want = snes.apply(theta, sigma, g_mu, g_sg, mask, 0.7, eta, smin, smax)
        got_t, got_s = dt.cpu().numpy(), ds.cpu().numpy()
        assert np.array_equal(got_t.view(np.uint32), theta.view(np.uint32)), step
        assert np.array_equal(got_s[~mask].view(np.uint32), sigma[~mask].view(np.uint32))
        ulps = np.abs(got_s.view(np.int32).astype(np.int64) - sigma_want.view(np.int32).astype(np.int64))
        assert ulps.max() <= 1, step                                          # the device exp vs NumPy's
        assert np.any(got_s[mask] == np.float32(smin)) and np.any(got_s[mask] == np.float32(smax))
        sigma = got_s.copy()                                                  # continue from the device state
        theta = got_t.copy()


# ---------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------
def _args(P, E=4, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=4, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.05, mutation_power_adversary=0.05,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
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
    if eng.separable:
        out["sigma"] = eng.sigma_cat.cpu().numpy().view(np.uint32)
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_engine_separable_deterministic():
    runs = []
    for _ in range(2):
        eng = _engine(64, **SNES_ALL)
        for _ in range(3):
            eng.step(sync=False)
        runs.append(_bits(eng))
    _same(*runs)
    sigma = runs[0]["sigma"].view(np.float32)
    moved = sigma[(sigma != 0) & (sigma != np.float32(0.05))]
    assert moved.size > 0 and moved.min() >= np.float32(0.001) and moved.max() <= np.float32(0.5)


def test_engine_separable_resume_bit_exact(tmp_path):
    full = _engine(64, **SNES_ALL)
    for _ in range(4):
        full.step(sync=False)
    first = _engine(64, **SNES_ALL)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "snes.pt")
    second = _engine(64, **SNES_ALL)
    second.load_state_dict(torch.load(tmp_path / "snes.pt", weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    _same(_bits(full), _bits(second))


def test_engine_explicit_isotropic_equals_an_engine_without_the_attribute():
    plain = _engine(64, adaptive=True)
    explicit = _engine(64, adaptive=True, es_distribution="isotropic", sigma_learning_rate=None)
    for _ in range(3):
        plain.step(sync=False)
        explicit.step(sync=False)
    _same(_bits(plain), _bits(explicit))
    assert plain.sigma_cat is None and explicit.sigma_cat is None


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
    eng = engine.ESEngine(_args(P, E, **SNES_ALL), dev, theta, comm=comm)
    eng.evaluate()
    eng.update()
    out = dict(rewards=np.stack([comm.all_gather_rows(eng.rewards[r], eng.shard).cpu().numpy() for r in ROLES]),
               grad=eng.grad_cat.cpu().numpy(), sigma=eng.sigma_cat.cpu().numpy())
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
def test_separable_sharded_over_two_gpus_equal_one_gpu():
    P, E = 386, 16                                 # 193 + 193 rows: the pair (192, 193) is cut by the boundary
    one = _launch(1, P, E, 29721)
    two = _launch(2, P, E, 29722)
    assert np.array_equal(one["rewards"], two["rewards"])
    scale = np.abs(one["grad"]).max()
    assert np.abs(one["grad"] - two["grad"]).max() <= 1e-5 * scale    # all-reduce summation order only
    np.testing.assert_allclose(two["sigma"], one["sigma"], rtol=1e-5, atol=0)
