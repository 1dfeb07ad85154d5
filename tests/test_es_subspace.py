"""Co-ES guided search on the host: the member formula and the coefficient stream of the oracle against scalar
restatements, flag validation, the drop-rule basis against numpy.linalg.qr, and the ES engine's guided-search path
with the checker backend (tests/es_subspace_backend.py): the estimate ring, k = 0 and alpha = 1 against the default
engine, resume, checkpoints and two gloo ranks."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_subspace as oss, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SUB = dict(es_subspace_dim=3, es_subspace_alpha=0.25)


# ---------------------------------------------------------------------------------------------------------------
# the member formula and the coefficients
# ---------------------------------------------------------------------------------------------------------------
def _scalar_member(theta, sigma, U, k_eff, alpha, z, c, sign):
    """One parameter at a time, one fp32 rounding per operation, straight from the header."""
    f = np.float32
    d = len(theta)
    A = f(math.sqrt(alpha))
    B = f(math.sqrt((1.0 - alpha) * d / k_eff)) if k_eff else f(0)
    out = np.empty(d, np.float32)
    for j in range(d):
        if B == 0:
            eps = f(z[j])
        else:
            s = f(0)
            for m in range(k_eff):
                s = f(s + f(f(U[m, j]) * f(c[m])))
            eps = f(f(A * f(z[j])) + f(B * s))
        dd = f(f(sigma) * eps)
        out[j] = f(theta[j] + (dd if sign > 0 else -dd))
    return out


@pytest.mark.parametrize("mirrored", [False, True], ids=["plain", "mirrored"])
@pytest.mark.parametrize("k_eff,alpha", [(3, 0.5), (5, 0.1), (1, 0.999), (0, 0.5), (4, 1.0)])
def test_member_formula_is_the_documented_one(mirrored, k_eff, alpha):
    rng = np.random.default_rng(3)
    D, n, row0 = 40, 5, 3
    pidx = np.array([j for j in range(D) if j % 7 != 3])            # a few copied (LayerNorm-like) entries
    theta = rng.standard_normal(D).astype(np.float32)
    U = rng.standard_normal((6, D)).astype(np.float32)
    z = rng.standard_normal((n, D)).astype(np.float32)
    c = rng.standard_normal((n, 6)).astype(np.float32)
    if mirrored:                                         # a pair shares its normals
        pair = (np.arange(row0, row0 + n) >> 1) - (row0 >> 1)
        z_pairs = z[:pair[-1] + 1]
        z, c = z_pairs[pair], c[pair]
    rows, eps = oss.perturb(theta, 0.05, U, k_eff, alpha, z, c, pidx, row0, mirrored)
    for r in range(n):
        sign = -1 if (mirrored and (row0 + r) & 1) else 1
        want = theta.copy()
        want[pidx] = _scalar_member(theta[pidx], 0.05, U[:, pidx], k_eff, alpha, z[r, pidx], c[r], sign)
        assert np.array_equal(rows[r], want), r
    if k_eff == 0 or alpha == 1.0:
        # B = 0: the members of the oracle's isotropic K5 restatements
        from oracle import es_options, ga_es
        iso = es_options.es_perturb_mirrored(theta, 0.05, z_pairs, pidx, row0, n) if mirrored else \
            ga_es.es_perturb(theta, 0.05, z, pidx)
        assert np.array_equal(rows, iso[0])


def test_variance_matches_the_isotropic_search():
    """E||eps||^2 = alpha d + (1 - alpha) d = d for an orthonormal U."""
    rng = np.random.default_rng(5)
    D, k, n = 200, 4, 4000
    U = np.linalg.qr(rng.standard_normal((D, k)))[0].T.astype(np.float32)
    z = rng.standard_normal((n, D)).astype(np.float32)
    c = rng.standard_normal((n, k)).astype(np.float32)
    _, eps = oss.perturb(np.zeros(D, np.float32), 1.0, U, k, 0.3, z, c, np.arange(D), 0, False)
    assert abs(np.mean(np.sum(eps.astype(np.float64) ** 2, axis=1)) / D - 1.0) < 0.02
    along = eps @ U.T                                                 # [n, k]
    assert np.allclose(np.var(along, axis=0), 0.3 + 0.7 * D / k, rtol=0.1)


def _scalar_coefficients(seed, role, gen, unit, k):
    k0, k1 = philox.split_seed(seed)
    out = []
    for m4 in range((k + 3) // 4):
        x = philox.philox4x32_10(np.uint32(m4), np.uint32(unit), np.uint32(gen),
                                 np.uint32(role | (oss.KIND_ES_SUBSPACE << 8)), k0, k1)
        z0, z1 = philox.box_muller(np.array([x[0]]), np.array([x[1]]))
        z2, z3 = philox.box_muller(np.array([x[2]]), np.array([x[3]]))
        out += [z0[0], z1[0], z2[0], z3[0]]
    return np.array(out[:k], np.float32)


@pytest.mark.parametrize("seed,role,gen,k", [(1870300, 0, 0, 1), (99, 2, 7, 16), (2 ** 40 + 3, 1, 2 ** 32 - 1, 32),
                                             (5, 0, 3, 7)])
def test_coefficients_are_the_documented_stream(seed, role, gen, k):
    units = np.array([0, 1, 17, 2 ** 32 - 1])
    c = oss.coefficients(seed, role, gen, units, k)
    assert c.dtype == np.float32 and c.shape == (4, k)
    for i, u in enumerate(units):
        assert np.array_equal(c[i], _scalar_coefficients(seed, role, gen, int(u), k))
    # c does not depend on k: a member's first k' coefficients are the same for every k >= k'
    assert np.array_equal(oss.coefficients(seed, role, gen, units, 32)[:, :k], c)
    # a stream of its own: not the K5 normals of the same member
    assert not np.array_equal(c, philox.normals(seed, philox.KIND_ES, role, gen, units, k))


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_subspace_flags_defaults_and_parsing():
    from coevonet_b200.engine import ES_SUBSPACE_DEFAULTS, es_subspace as validate
    a = _cli(["--algorithm=ES"])
    assert (a.es_subspace_dim, a.es_subspace_alpha) == (0, None)
    assert validate(a) == ES_SUBSPACE_DEFAULTS
    assert validate(types.SimpleNamespace(population=4)) == ES_SUBSPACE_DEFAULTS           # attributes absent
    assert validate(_cli(["--algorithm=ES", "--es_subspace_dim=16"])) == {"es_subspace_dim": 16,
                                                                        "es_subspace_alpha": 0.5}
    assert validate(_cli(["--algorithm=ES", "--es_subspace_dim=32", "--es_subspace_alpha=1"])) == \
        {"es_subspace_dim": 32, "es_subspace_alpha": 1.0}
    # with the other Co-ES options
    assert validate(_cli(["--algorithm=ES", "--es_subspace_dim=4", "--mirrored_sampling", "--es_optimizer=adam",
                          "--es_hof_size=2", "--fitness_shaping=centered_rank"]))["es_subspace_dim"] == 4


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=GA", "--es_subspace_dim=4"], "GA"),
    (["--algorithm=GA", "--es_subspace_dim=4", "--es_subspace_alpha=0.5"], "GA"),
    (["--algorithm=ES", "--es_subspace_dim=33"], r"\[0, 32\]"),
    (["--algorithm=ES", "--es_subspace_dim=-1"], r"\[0, 32\]"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--es_subspace_alpha=0"], r"\(0, 1\]"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--es_subspace_alpha=1.5"], r"\(0, 1\]"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--es_subspace_alpha=-0.2"], r"\(0, 1\]"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--es_subspace_alpha=nan"], r"\(0, 1\]"),
    (["--algorithm=ES", "--es_subspace_alpha=0.5"], "needs es_subspace_dim"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--es_distribution=separable"], "separable"),
    (["--algorithm=ES", "--es_subspace_dim=4", "--regenerate_noise"], "regenerate_noise"),
])
def test_subspace_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_ga_engine_refuses_the_subspace_options():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="GA"):
        engine.GAEngine(_args(4, algorithm="GA", es_subspace_dim=2), "cpu", {}, {}, {}, kernels=_backend())


# ---------------------------------------------------------------------------------------------------------------
# the basis
# ---------------------------------------------------------------------------------------------------------------
def _check_basis(D, kept, tol_orth=1e-5, tol_proj=1e-4):
    """U of the oracle against numpy.linalg.qr of the estimates it should keep (newest first)."""
    U = oss.basis(D)
    assert U.shape == (len(kept), D.shape[1])
    if not kept:
        return U
    U64 = U.astype(np.float64)
    assert np.max(np.abs(U64 @ U64.T - np.eye(len(kept)))) <= tol_orth
    Q = np.linalg.qr(D[kept].astype(np.float64).T)[0]
    # projectors of equal rank: max |U^T U - Q Q^T| <= ||U^T U - Q Q^T||_2 = ||(I - Q Q^T) U^T||_2
    assert np.linalg.norm(U64.T - Q @ (Q.T @ U64.T), 2) <= tol_proj
    # the first direction is the newest kept estimate
    v = D[kept[0]] / np.linalg.norm(D[kept[0]])
    assert abs(abs(float(U64[0] @ v)) - 1.0) < 1e-6
    return U


def test_basis_of_random_estimates():
    rng = np.random.default_rng(11)
    D = (rng.standard_normal((8, 600)) * rng.uniform(1e-3, 1e2, (8, 1))).astype(np.float32)
    _check_basis(D, list(range(8)))


def test_basis_drops_dependent_and_zero_estimates():
    rng = np.random.default_rng(12)
    a, b = rng.standard_normal((2, 500)).astype(np.float32)
    D = np.stack([a, np.zeros(500, np.float32), b, (2 * a - 3 * b).astype(np.float32), -a,
                  rng.standard_normal(500).astype(np.float32)])
    _check_basis(D, [0, 2, 5])
    assert oss.basis(np.zeros((4, 100), np.float32)).shape == (0, 100)       # all ties: nothing to search along


@pytest.mark.parametrize("bad", [np.nan, np.inf], ids=["nan", "inf"])
def test_basis_drops_a_non_finite_estimate(bad):
    rng = np.random.default_rng(15)
    D = rng.standard_normal((4, 300)).astype(np.float32)
    D[1, 7] = bad
    U = _check_basis(D, [0, 2, 3])
    assert np.all(np.isfinite(U))


def test_basis_of_nearly_parallel_estimates():
    rng = np.random.default_rng(13)
    a, e = rng.standard_normal((2, 800))
    D = np.stack([a, a + 1e-6 * e, a + 1e-2 * e]).astype(np.float32)
    # residual 1e-6 of its norm: dropped; 1e-2: kept
    _check_basis(D, [0, 2])


def test_ring_basis_keeps_segments_apart():
    """Each role gets its own basis over its Linear entries; everything else stays 0."""
    from coevonet_b200 import layout
    from oracle import layout as olayout
    rng = np.random.default_rng(14)
    dims = [layout.OBS_DIM[r] for r in ROLES]
    pitches = [layout.fc_pitch(d) for d in dims]
    n = sum(pitches)
    ring = oss.Ring(4, n)
    segs, start = [], 0
    for d, p in zip(dims, pitches):
        segs.append((start, start + p, olayout.fc_perturbable_index(d)))
        start += p
    mask = np.zeros(n, bool)
    for s0, _, pidx in segs:
        mask[s0 + pidx] = True
    for g in range(6):
        row = np.where(mask, rng.standard_normal(n), 0).astype(np.float32)
        if g == 3:
            row[segs[1][0]:segs[1][1]] = 0                            # agent_1's estimate is zero this generation
        ring.append(row)
    U, ke = oss.ring_basis(ring.rows, ring.newest, ring.filled, segs)
    assert ke == [4, 3, 4]
    assert not np.any(U[:, ~mask])
    for (s0, s1, pidx), kk in zip(segs, ke):
        _check_basis(ring.newest_first()[:, s0 + pidx], [a for a in range(4) if not (s0 == segs[1][0] and a == 2)])
        assert not np.any(U[kk:, s0:s1])


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import es_subspace_backend
    return es_subspace_backend


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


def test_zero_dimension_issues_the_default_calls():
    logs = []
    for kw in ({}, {"es_subspace_dim": 0}):
        log = _Log()
        eng = _engine(4, kernels=log, **kw)
        for _ in range(2):
            eng.step()
        assert eng.subspace_ring is None and eng.history[0]["subspace_rank"] is None
        logs.append(log.calls)
    assert logs[0] == logs[1] and "es_perturb" in logs[0]
    assert not any("subspace" in c for c in logs[0])


@pytest.mark.parametrize("mirrored", [False, True], ids=["plain", "mirrored"])
def test_alpha_one_equals_the_default_engine(mirrored):
    a = _engine(4, mirrored_sampling=mirrored)
    b = _engine(4, mirrored_sampling=mirrored, es_subspace_dim=2, es_subspace_alpha=1.0)
    for g in range(3):
        assert a.step() == b.step()
        for r in ROLES:
            assert np.array_equal(a.history[g]["rewards"][r], b.history[g]["rewards"][r])
            assert np.array_equal(a.history[g]["delta"][r], b.history[g]["delta"][r])
        assert torch.equal(a.theta_cat, b.theta_cat)
    assert b.history[2]["subspace_rank"] == {r: 2 for r in ROLES}
    assert torch.equal(a.gstate, b.gstate)


def test_ring_and_basis_follow_the_oracle():
    """k = 3 over k + 2 = 5 generations: the ring, head, filled, U and k_eff after every generation against the
    oracle's ring and basis, and the members of every generation against the member formula with that basis."""
    from coevonet_b200 import layout
    from oracle import layout as olayout
    k = 3
    eng = _engine(4, es_subspace_dim=k, es_subspace_alpha=0.3, mirrored_sampling=True)
    ring = oss.Ring(k, eng.theta_cat.numel())
    segs = [(o, o + p, olayout.fc_perturbable_index(layout.OBS_DIM[r])) for r, (o, p) in eng.cols.items()]
    U = np.zeros((k, eng.theta_cat.numel()), np.float32)
    ke = [0, 0, 0]
    for g in range(k + 2):
        theta = eng.theta_cat.numpy().copy()
        eng.step()
        assert eng.history[g]["subspace_rank"] == {r: min(g + 1, k) for r in ROLES}
        for i, role in enumerate(ROLES):                 # this generation's members used the previous basis
            o, p = eng.cols[role]
            in_dim = layout.OBS_DIM[role]
            D = layout.fc_dim(in_dim)
            z = _backend()._normals(99, role, g, 0, 4, D, True)
            c = oss.coefficients(99, i, g, np.arange(4) >> 1, k)
            rows, _ = oss.perturb(theta[o:o + D], eng.args.mutation_power_agent_0 if i == 0 else
                                  eng.args.mutation_power_agent_1 if i == 1 else eng.args.mutation_power_adversary,
                                  U[:, o:o + D], ke[i], 0.3, z, c, olayout.fc_perturbable_index(in_dim), 0, True)
            assert np.array_equal(eng.members[role].numpy()[:, :D], rows), (g, role)
        ring.append(np.concatenate([eng.history[g]["delta"][r] for r in ROLES]))
        assert (eng.subspace_head, eng.subspace_filled) == (ring.head, ring.filled)
        assert np.array_equal(eng.subspace_ring.numpy(), ring.rows)
        U, ke = oss.ring_basis(ring.rows, ring.newest, ring.filled, segs)
        assert np.array_equal(eng.subspace_U.numpy(), U) and eng.subspace_keff.tolist() == ke


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(SUB, record_history=False)
    full = _engine(4, **kw)
    for _ in range(5):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "sub.pt")
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(tmp_path / "sub.pt", weights_only=False))
    assert torch.equal(second.subspace_U, first.subspace_U) and torch.equal(second.subspace_keff, first.subspace_keff)
    for _ in range(3):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.theta_cat, full.theta_cat)
    assert torch.equal(second.subspace_ring, full.subspace_ring)
    assert torch.equal(second.subspace_U, full.subspace_U)
    assert (second.subspace_head, second.subspace_filled) == (full.subspace_head, full.subspace_filled)


def test_resume_refuses_other_subspace_settings():
    sub = _engine(4, record_history=False, **SUB)
    sub.step(sync=False)
    sd = sub.state_dict()
    assert sd["es_subspace"] == SUB and sd["subspace_filled"] == 1
    with pytest.raises(ValueError, match="guided search"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="guided search"):
        _engine(4, record_history=False, es_subspace_dim=3).load_state_dict(sd)          # alpha 0.5 != 0.25
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    assert plain.state_dict()["es_subspace"] == {"es_subspace_dim": 0, "es_subspace_alpha": None}
    with pytest.raises(ValueError, match="guided search"):
        _engine(4, record_history=False, **SUB).load_state_dict(plain.state_dict())
    # a checkpoint without the settings (written before they existed) loads as k = 0
    old = plain.state_dict()
    del old["es_subspace"]
    fresh = _engine(4, record_history=False)
    fresh.load_state_dict(old)
    assert torch.equal(fresh.theta_cat, plain.theta_cat)
    with pytest.raises(ValueError, match="guided search"):
        _engine(4, record_history=False, **SUB).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **SUB)
    evs = [eng.step() for _ in range(3)]
    q.put(dict(rank=rank, evs=np.asarray(evs),
               rewards=np.stack([eng.history[g]["rewards"][r] for g in range(3) for r in ROLES]),
               ranks=[eng.history[g]["subspace_rank"] for g in range(3)],
               theta=eng.theta_cat.numpy().copy(), ring=eng.subspace_ring.numpy().copy(),
               U=eng.subspace_U.numpy().copy()))
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
def test_subspace_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows; the ring and the basis are replicated."""
    P = 5
    single = _launch(1, P, 29661)[0]
    two = _launch(2, P, 29662)
    for o in two:
        assert o["ranks"] == single["ranks"]
        # generation 0 draws the same members from the same founders
        assert np.array_equal(o["rewards"][:3], single["rewards"][:3])
        np.testing.assert_allclose(o["rewards"], single["rewards"], rtol=1e-12, atol=0)
        # the two ranks' partial updates are added in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["ring"], single["ring"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["U"], single["U"], rtol=0, atol=1e-4)
    for k in ("theta", "ring", "U", "rewards"):
        assert np.array_equal(two[0][k], two[1][k])                    # replicas agree bit for bit
