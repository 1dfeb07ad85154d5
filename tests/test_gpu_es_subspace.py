"""Co-ES guided search on the GPU: the subspace K5 against the oracle's member formula bit for bit (given the kernel's
own normals), the isotropic members when k_eff = 0 or alpha = 1, the basis kernel against numpy.linalg.qr, the
variance of the search directions, engine determinism, resume and defaults, and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_subspace as oss

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 31337


def _layout():
    from coevonet_b200 import layout
    from oracle import layout as olayout
    dims = [layout.OBS_DIM[r] for r in ROLES]
    pitches = [layout.fc_pitch(d) for d in dims]
    offs = np.cumsum([0] + pitches[:-1]).tolist()
    segs = [(o, o + p, olayout.fc_perturbable_index(d)) for o, p, d in zip(offs, pitches, dims)]
    return dims, pitches, offs, segs


def _ring(k, filled, seed=1):
    """A ring of estimates on the Linear entries of the three roles, with a zero estimate and a nearly parallel
    one in agent_1's segment and an exactly dependent one in the adversary's."""
    dims, pitches, offs, segs = _layout()
    n = sum(pitches)
    rng = np.random.default_rng(seed)
    ring = oss.Ring(k, n)
    for g in range(filled):
        row = np.zeros(n, np.float32)
        for s0, _, pidx in segs:
            row[s0 + pidx] = rng.standard_normal(len(pidx)) * 10.0 ** rng.uniform(-4, 0)
        ring.append(row)
    rows = ring.rows
    if filled >= 4:
        s0, s1, pidx = segs[1]
        rows[ring.newest, s0:s1] = 0                                    # all-tied ranks: a zero estimate
        prev = (ring.newest - 1) % k
        rows[(ring.newest - 2) % k, s0 + pidx] = rows[prev, s0 + pidx] * np.float32(1 + 1e-7)  # nearly parallel
        s0, s1, pidx = segs[2]
        a, b = (ring.newest - 1) % k, (ring.newest - 2) % k
        rows[(ring.newest - 3) % k, s0 + pidx] = (rows[a, s0 + pidx] - 2 * rows[b, s0 + pidx]).astype(np.float32)
    return ring, segs


def _basis(ring, dims):
    from coevonet_b200 import ops
    return ops.es_subspace_basis(torch.from_numpy(ring.rows).cuda(), ring.newest, ring.filled, dims)


@pytest.mark.parametrize("k,filled", [(1, 1), (4, 2), (6, 6), (16, 16), (32, 9)])
def test_basis_kernel_matches_qr_and_is_deterministic(k, filled):
    dims, _, _, segs = _layout()
    ring, _ = _ring(k, filled)
    U, ke = _basis(ring, dims)
    U2, ke2 = _basis(ring, dims)
    assert torch.equal(U, U2) and torch.equal(ke, ke2)                  # deterministic
    U, ke = U.cpu().numpy(), ke.cpu().tolist()
    Uo, keo = oss.ring_basis(ring.rows, ring.newest, ring.filled, segs)
    assert ke == keo
    if filled >= 4:
        assert ke == [filled, filled - 2, filled - 1]
    mask = np.zeros(U.shape[1], bool)
    for si, ((s0, s1, pidx), kk) in enumerate(zip(segs, ke)):
        mask[s0 + pidx] = True
        Us = U[:kk, s0 + pidx].astype(np.float64)
        assert not np.any(U[kk:, s0:s1])
        assert np.max(np.abs(Us @ Us.T - np.eye(kk))) <= 1e-5
        D = ring.newest_first()[:, s0 + pidx].astype(np.float64)
        kept = list(range(filled))                                    # newest first; the drops of _ring
        if filled >= 4:
            kept = {0: kept, 1: [1] + kept[3:], 2: kept[:3] + kept[4:]}[si]
        assert len(kept) == kk
        Q = np.linalg.qr(D[kept].T)[0]
        assert np.linalg.norm(Us.T - Q @ (Q.T @ Us.T), 2) <= 1e-4
        np.testing.assert_allclose(Us, Uo[:kk, s0 + pidx], rtol=0, atol=1e-5)
    assert not np.any(U[:, ~mask])


@pytest.mark.parametrize("bad", [np.nan, np.inf], ids=["nan", "inf"])
def test_basis_kernel_drops_a_non_finite_estimate(bad):
    """A non-finite estimate is dropped and never reaches U: its role keeps the basis of the other estimates."""
    dims, _, _, segs = _layout()
    ring, _ = _ring(6, 5)
    s0, _, pidx = segs[0]
    ring.rows[(ring.newest - 1) % 6, s0 + pidx[11]] = bad
    U, ke = _basis(ring, dims)
    U, ke = U.cpu().numpy(), ke.cpu().tolist()
    Uo, keo = oss.ring_basis(ring.rows, ring.newest, ring.filled, segs)
    assert ke == keo and ke[0] == 4
    assert np.all(np.isfinite(U))
    np.testing.assert_allclose(U, Uo, rtol=0, atol=1e-5)


def test_basis_kernel_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    dims, pitches, _, _ = _layout()
    ring = torch.zeros((4, sum(pitches)), device="cuda")
    for newest, filled in ((4, 1), (0, 5), (-1, 1)):
        with pytest.raises(_lib.CevError):
            ops.es_subspace_basis(ring, newest, filled, dims)
    with pytest.raises(_lib.CevError):
        ops.es_subspace_basis(torch.zeros((33, sum(pitches)), device="cuda"), 0, 1, dims)


def _role_inputs(role, k, filled, seed=2):
    """theta of the role and its columns of a basis computed by the kernel (row stride len(theta_cat))."""
    from coevonet_b200 import layout, ops
    dims, _, offs, _ = _layout()
    ring, _ = _ring(k, filled, seed)
    U, ke = _basis(ring, dims)
    i = ROLES.index(role)
    o, p = offs[i], layout.fc_pitch(dims[i])
    theta = ops.fc_init(dims[i], 5, role, 0, 1, "cuda")[0]
    return theta, U[:, o:o + p], ke[i:i + 1], dims[i]


def _oracle_rows(theta, sigma, U, k_eff, alpha, noise, coef, in_dim):
    """The member formula given the kernel's signed normals (s z, s c): the odd member of a mirrored pair is the
    formula at (-z, -c), which negates eps exactly."""
    from coevonet_b200 import layout
    from oracle import layout as olayout
    D = layout.fc_dim(in_dim)
    rows, _ = oss.perturb(theta.cpu().numpy()[:D], sigma, U.cpu().numpy()[:, :D], k_eff, alpha,
                          noise.cpu().numpy()[:, :D], coef.cpu().numpy(), olayout.fc_perturbable_index(in_dim), 0,
                          False)
    return rows


@pytest.mark.parametrize("mirrored", [False, True], ids=["plain", "mirrored"])
@pytest.mark.parametrize("role,k,filled,alpha", [("agent_0", 5, 5, 0.5), ("adversary_0", 16, 7, 0.2),
                                                 ("agent_1", 32, 32, 0.9)])
def test_subspace_k5_matches_the_oracle_bit_for_bit_across_a_shard_boundary(mirrored, role, k, filled, alpha):
    from coevonet_b200 import layout, ops
    theta, U, ke, in_dim = _role_inputs(role, k, filled)
    pitch = layout.fc_pitch(in_dim)
    sigma, P, cut = 0.05, 70, 33                                      # the cut splits pair 16
    full = ops.es_perturb_subspace(theta, in_dim, sigma, U, ke, alpha, SEED, role, 3, 0, P, mirrored=mirrored)
    parts = []
    for row0, n in ((0, cut), (cut, P - cut)):
        noise = torch.empty((n, pitch), device="cuda")
        coef = torch.empty((n, k), device="cuda")
        rows = ops.es_perturb_subspace(theta, in_dim, sigma, U, ke, alpha, SEED, role, 3, row0, n, mirrored=mirrored,
                                       noise_out=noise, coef_out=coef)
        want = _oracle_rows(theta, sigma, U, int(ke.item()), alpha, noise, coef, in_dim)
        got = rows.cpu().numpy()
        D = layout.fc_dim(in_dim)
        assert np.array_equal(got[:, :D], want) and not np.any(got[:, D:])
        parts.append((rows, noise, coef))
    assert torch.equal(torch.cat([p[0] for p in parts]), full)
    coef = torch.cat([p[2] for p in parts]).cpu().numpy()
    units = np.arange(P) >> 1 if mirrored else np.arange(P)
    sign = np.where((np.arange(P) & 1) & mirrored, -1, 1)[:, None]
    c = oss.coefficients(SEED, layout.ROLE_ID[role], 3, units, k) * sign
    np.testing.assert_allclose(coef, c, rtol=0, atol=2e-5)          # the documented stream (libm vs MUFU)
    if mirrored:                                                      # a pair shares its normals, with opposite signs
        noise = torch.cat([p[1] for p in parts])
        assert torch.equal(noise[1::2], -noise[0::2]) and np.array_equal(coef[1::2], -coef[0::2])


@pytest.mark.parametrize("mirrored", [False, True], ids=["plain", "mirrored"])
@pytest.mark.parametrize("case", ["k_eff_0", "alpha_1"])
def test_isotropic_members_when_the_subspace_term_vanishes(mirrored, case):
    from coevonet_b200 import ops
    role = "adversary_0"
    theta, U, ke, in_dim = _role_inputs(role, 8, 8)
    alpha = 1.0 if case == "alpha_1" else 0.3
    if case == "k_eff_0":
        ke = torch.zeros(1, dtype=torch.int32, device="cuda")
    sigma = torch.tensor([0.05], dtype=torch.float64, device="cuda")   # the engine's device sigma
    iso = ops.es_perturb_mirrored if mirrored else ops.es_perturb
    for row0, n in ((0, 64), (7, 41)):
        got = ops.es_perturb_subspace(theta, in_dim, sigma, U, ke, alpha, SEED, role, 2, row0, n, mirrored=mirrored)
        assert torch.equal(got, iso(theta, in_dim, sigma, SEED, role, 2, row0, n))


def test_search_directions_have_the_documented_variance():
    """8,192 members, k_eff = 16, alpha = 0.25: along each basis direction the variance of eps is
    alpha + (1 - alpha) d / k_eff, along random directions orthogonal to U it is alpha.  The sample variance of n
    normals has a relative standard deviation of sqrt(2 / n) = 1.6 %: the tolerance is 5 of those, 7.8 %."""
    from coevonet_b200 import layout
    from coevonet_b200 import ops
    from oracle import layout as olayout
    role, k, alpha, sigma, P = "agent_0", 16, 0.25, 0.01, 8192
    theta, U, ke, in_dim = _role_inputs(role, k, k, seed=4)
    assert int(ke.item()) == k
    pidx = olayout.fc_perturbable_index(in_dim)
    d = len(pidx)
    Ud = U.cpu().numpy()[:, pidx].astype(np.float64)
    rng = np.random.default_rng(9)
    W = rng.standard_normal((8, d))
    W -= (W @ Ud.T) @ Ud                                              # orthogonal to the subspace
    W /= np.linalg.norm(W, axis=1, keepdims=True)
    dirs = torch.from_numpy(np.concatenate([Ud, W]).T).cuda()        # [d, k + 8]
    th = theta[torch.from_numpy(pidx).cuda()].double()
    proj = []
    for row0 in range(0, P, 1024):
        rows = ops.es_perturb_subspace(theta, in_dim, sigma, U, ke, alpha, SEED, role, 0, row0, 1024)
        eps = (rows[:, torch.from_numpy(pidx).cuda()].double() - th) / sigma
        proj.append(eps @ dirs)
    var = torch.cat(proj).var(dim=0).cpu().numpy()
    tol = 5 * np.sqrt(2.0 / P)
    np.testing.assert_allclose(var[:k], alpha + (1 - alpha) * d / k, rtol=tol)
    np.testing.assert_allclose(var[k:], alpha, rtol=tol)


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


def _bits(eng):
    eng.check_status()
    out = {"theta": eng.theta_cat.cpu().numpy().view(np.uint32), "gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["rew_" + r] = eng.rewards[r].cpu().numpy()
    if eng.subspace_ring is not None:
        out["ring"] = eng.subspace_ring.cpu().numpy().view(np.uint32)
        out["U"] = eng.subspace_U.cpu().numpy().view(np.uint32)
        out["keff"] = eng.subspace_keff.cpu().numpy()
    return out


def _same(a, b, keys=None):
    for k in keys or a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("mirrored", [False, True], ids=["plain", "mirrored"])
def test_defaults_and_alpha_one_equal_the_default_engine(mirrored):
    plain = _engine(64, mirrored_sampling=mirrored)
    zero = _engine(64, mirrored_sampling=mirrored, es_subspace_dim=0)
    one = _engine(64, mirrored_sampling=mirrored, es_subspace_dim=4, es_subspace_alpha=1.0)
    keys = ["theta", "gstate"] + [p + r for p in ("fit_", "rew_") for r in ROLES]
    for _ in range(3):
        for e in (plain, zero, one):
            e.step(sync=False)
        ref = _bits(plain)
        _same(ref, _bits(zero), keys)
        _same(ref, _bits(one), keys)
    assert zero.subspace_ring is None
    assert _bits(one)["keff"].tolist() == [3, 3, 3]


def test_subspace_engine_deterministic_and_resume_bit_exact(tmp_path):
    kw = dict(es_subspace_dim=3, es_subspace_alpha=0.5, mirrored_sampling=True, fitness_shaping="centered_rank",
              es_optimizer="adam", learning_rate=0.01)
    runs = []
    for _ in range(2):
        eng = _engine(64, **kw)
        for _ in range(5):
            eng.step(sync=False)
        runs.append(_bits(eng))
    _same(*runs)
    assert runs[0]["keff"].tolist() == [3, 3, 3]
    first = _engine(64, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "sub.pt")
    second = _engine(64, **kw)
    second.load_state_dict(torch.load(tmp_path / "sub.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    _same(runs[0], _bits(second))


def test_subspace_moves_the_members_off_the_isotropic_rows():
    """With k > 0 and alpha < 1 the members of generation 1 differ from the isotropic ones; those of generation 0
    (an empty ring, k_eff = 0) do not."""
    plain = _engine(32)
    sub = _engine(32, es_subspace_dim=2)
    plain.evaluate()
    sub.evaluate()
    for r in ROLES:
        assert torch.equal(plain.members[r], sub.members[r])
    plain.update()
    sub.update()
    plain.gen += 1
    sub.gen += 1
    plain.evaluate()
    sub.evaluate()
    for r in ROLES:
        assert not torch.equal(plain.members[r], sub.members[r])


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
    eng = engine.ESEngine(_args(P, E, es_subspace_dim=4, mirrored_sampling=True), dev, theta, comm=comm)
    for _ in range(3):
        eng.step(sync=False)
    out = dict(theta=eng.theta_cat.cpu().numpy(), ring=eng.subspace_ring.cpu().numpy(),
               U=eng.subspace_U.cpu().numpy(), keff=eng.subspace_keff.cpu().numpy())
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
def test_subspace_sharded_over_two_gpus_equal_one_gpu():
    P, E = 386, 16                                 # 193 + 193 rows: the shard boundary cuts pair 96
    one = _launch(1, P, E, 29741)[0]
    two = _launch(2, P, E, 29742)
    for k in ("theta", "ring", "U", "keff"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree
    for o in two:
        assert np.array_equal(o["keff"], one["keff"])
        # the all-reduce adds the ranks' partial updates in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], one["theta"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(o["ring"], one["ring"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(o["U"], one["U"], rtol=0, atol=1e-3)
