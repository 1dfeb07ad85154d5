"""Co-ES LM-MA-ES on the host: the compact transform against the sequential one, the constants, the restated algorithm
as an optimiser (linear, sphere, rotated ellipsoid), flag validation, and the ES engine's LM-MA-ES path on the checker
backend (tests/es_lmma_backend.py): the default call log, the engine against the oracle, resume, checkpoints and two
gloo ranks."""
import math
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_lmma as olm

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
LM = dict(es_distribution="lmma", es_lmma_memory=3, learning_rate=1.0)


# ---------------------------------------------------------------------------------------------------------------
# the transform and the constants
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k,m", [(1, 1), (2, 8), (5, 8), (8, 8), (16, 32), (32, 32)])
@pytest.mark.parametrize("collinear", [False, True], ids=["random", "near_collinear"])
def test_compact_transform_equals_the_sequential_one(k, m, collinear):
    rng = np.random.default_rng(k + 100 * m)
    n = 300
    M = rng.standard_normal((m, n)) * rng.uniform(0.1, 10, (m, 1))
    if collinear and m > 1:
        M[1] = M[0] * (1 + 1e-9) + 1e-9 * rng.standard_normal(n)
    z = rng.standard_normal((4, n))
    c_d = olm.constants(64, n, m)["c_d"]
    alpha, beta = olm.transform_compact(z @ M[:k].T, M @ M.T, k, c_d)
    d = alpha * z + beta @ M[:k]
    want = olm.transform_sequential(M, z, k, c_d)
    assert np.max(np.abs(d - want)) <= 1e-12 * max(1.0, np.max(np.abs(want)))
    assert alpha == olm.alpha_of(k, c_d)


def test_constants_match_their_formulas_and_the_engine():
    from coevonet_b200 import engine
    for lam, n, m in ((1024, 138245, 8), (7, 64, 3), (2, 10, 1)):
        c = olm.constants(lam, n, m)
        mu = lam // 2
        assert c["mu"] == mu and len(c["w"]) == mu
        assert abs(c["w"].sum() - 1.0) < 1e-15 and np.all(np.diff(c["w"]) < 0)
        assert math.isclose(c["mu_w"], 1.0 / np.sum(c["w"] ** 2), rel_tol=1e-15)
        assert c["c_sigma"] == 2 * lam / n
        for j in range(m):
            assert math.isclose(c["c_d"][j], 1 / (1.5 ** j * n), rel_tol=1e-15)
            assert math.isclose(c["c_c"][j], lam / (4 ** j * n), rel_tol=1e-15)
        e = engine.lmma_constants(lam, n, m)
        assert e["mu"] == mu and e["c_d"] == c["c_d"] and e["c_c"] == c["c_c"] and e["c_sigma"] == c["c_sigma"]
        np.testing.assert_allclose(e["w"], c["w"], rtol=1e-15)
        assert e["alpha"] == [olm.alpha_of(k, c["c_d"]) for k in range(m + 1)]


# ---------------------------------------------------------------------------------------------------------------
# the restated algorithm is a working LM-MA-ES
# ---------------------------------------------------------------------------------------------------------------
def test_sigma_grows_on_a_linear_function():
    _, sigma, _ = olm.minimize(lambda x: float(x[0]), 64, 16, 8, 1e-3, 100, np.random.default_rng(1))
    assert sigma > 10.0                                   # 1e-3 -> ~84 in 100 generations


def test_converges_on_the_sphere():
    _, _, hist = olm.minimize(lambda x: float(x @ x), 64, 16, 8, 1.0, 2000, np.random.default_rng(1), x0=np.ones(64),
                              target=1e-10)
    assert hist[-1] <= 1e-10 and len(hist) < 800          # 487 generations with this seed


def test_vectors_help_on_a_rotated_ill_conditioned_ellipsoid():
    """n = 64, condition 1e6, lam = 16, 2e4 generations from x = 1: with these constants neither run reaches 1e-8 in
    that budget, but m = 8 ends more than 1000x lower than m = 0 (plain CSA-ES; ~1e3 vs ~0.6 over three seeds)."""
    n = 64
    rng = np.random.default_rng(0)
    Q = np.linalg.qr(rng.standard_normal((n, n)))[0]
    scale = 10.0 ** (6 * np.arange(n) / (n - 1))

    def f(x):
        y = Q @ x
        return float(np.sum(scale * y * y))
    ends = {}
    for m in (0, 8):
        ends[m] = olm.minimize(f, n, 16, m, 1.0, 20000, np.random.default_rng(0), x0=np.ones(n), target=1e-8)[2][-1]
    assert ends[8] * 1000 < ends[0]


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_lmma_flags_defaults_and_parsing():
    from coevonet_b200.engine import ES_DISTRIBUTION_DEFAULTS, es_distribution as validate
    a = _cli(["--algorithm=ES"])
    assert a.es_lmma_memory is None and validate(a) == ES_DISTRIBUTION_DEFAULTS
    assert validate(_cli(["--algorithm=ES", "--es_distribution=lmma"]))["es_lmma_memory"] == 8
    assert validate(_cli(["--algorithm=ES", "--es_distribution=lmma", "--es_lmma_memory=32", "--es_hof_size=2",
                          "--fitness_sharing", "--learning_rate=1.0"]))["es_lmma_memory"] == 32


@pytest.mark.parametrize("argv,match", [
    (["--es_lmma_memory=4"], "needs es_distribution 'lmma'"),
    (["--es_distribution=separable", "--es_lmma_memory=4"], "needs es_distribution 'lmma'"),
    (["--es_distribution=lmma", "--es_lmma_memory=0"], r"\[1, 32\]"),
    (["--es_distribution=lmma", "--es_lmma_memory=33"], r"\[1, 32\]"),
    (["--es_distribution=lmma", "--es_optimizer=adam"], "own step"),
    (["--es_distribution=lmma", "--l2_coeff=0.01"], "own step"),
    (["--es_distribution=lmma", "--adaptive"], "cumulative step-size"),
    (["--es_distribution=lmma", "--fitness_shaping=centered_rank"], "log weights"),
    (["--es_distribution=lmma", "--mirrored_sampling"], "mirrored"),
    (["--es_distribution=lmma", "--es_subspace_dim=4"], "es_subspace_dim"),
    (["--es_distribution=lmma", "--fitness_shaping=centered_rank", "--es_novelty_weight=0.5"], "log weights"),
    (["--es_distribution=lmma", "--sigma_learning_rate=0.1"], "separable"),
    (["--es_distribution=lmma", "--population=68611"], "c_sigma"),
    (["--algorithm=GA", "--es_distribution=lmma"], "GA"),
])
def test_lmma_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8", "--algorithm=ES"] + argv if not any("GA" in x for x in argv) else argv)


def test_novelty_refusal_and_largest_population():
    from coevonet_b200 import engine
    a = types.SimpleNamespace(population=8, es_distribution="lmma", fitness_shaping="none", es_novelty_weight=0.5)
    with pytest.raises(ValueError, match="es_novelty_weight"):
        engine.es_distribution(a)
    assert engine.LMMA_MIN_DIM == 137221
    engine.es_distribution(types.SimpleNamespace(population=68610, es_distribution="lmma"))
    # the guided-search refusal names the distribution given
    with pytest.raises(ValueError, match="'lmma'"):
        engine.es_subspace(types.SimpleNamespace(population=8, es_distribution="lmma", es_subspace_dim=2))


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import es_lmma_backend
    return es_lmma_backend


class _Log:
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
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_es_subspace
    return test_es_subspace._args(P, record_history, **opts)


def _engine(P, comm=None, kernels=None, **kw):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_es_subspace
    from coevonet_b200 import engine
    return engine.ESEngine(_args(P, **kw), "cpu", test_es_subspace._theta(), kernels=kernels or _backend(), comm=comm)


def test_default_distribution_issues_the_default_calls():
    logs = []
    for kw in ({}, {"es_distribution": "isotropic"}):
        log = _Log()
        eng = _engine(4, kernels=log, **kw)
        for _ in range(2):
            eng.step()
        assert eng.lmma_M is None and eng.history[0]["lmma"] is None
        logs.append(log.calls)
    assert logs[0] == logs[1] and "es_perturb" in logs[0]
    assert not any("lmma" in c for c in logs[0])


def test_engine_follows_the_oracle_with_the_hall_of_fame_and_fitness_sharing():
    from coevonet_b200 import _lib, layout
    from oracle import layout as olayout
    P, m = 6, 3
    eng = _engine(P, es_hof_size=3, es_hof_opponents=2, **LM)
    assert eng.args.fitness_sharing
    for g in range(4):
        th, M, p, G = (x.numpy().copy() for x in (eng.theta_cat, eng.lmma_M, eng.lmma_p, eng.lmma_G))
        sig = eng.gstate[_lib.GS_SIGMA:_lib.GS_SIGMA + 3].numpy().copy()
        eng.step()
        k = min(g, m)
        assert eng.history[g]["lmma"]["agent_1"]["k_eff"] == k
        for i, role in enumerate(ROLES):
            o, pitch = eng.cols[role]
            in_dim = layout.OBS_DIM[role]
            D = layout.fc_dim(in_dim)
            pidx = olayout.fc_perturbable_index(in_dim)
            c = eng.lmma_const[role]              # equal to olm.constants (test above) to the last bit or so
            z = _backend()._z(99, role, g, 0, P, in_dim)
            s = olm.project(M[:, o:o + D], z, k) if k else np.zeros((P, 0))
            alpha, b = olm.transform_compact(s, G[i], k, c["c_d"])
            b32 = b.astype(np.float32)
            rows = olm.perturb(th[o:o + D], np.float32(sig[i]), M[:, o:o + D], b32, alpha, z, pidx)
            assert np.array_equal(eng.members[role].numpy()[:, :D], rows), (g, role)
            ids = np.argsort(-eng.fitness[role].numpy(), kind="stable")[:c["mu"]]
            zfull = np.zeros((P, pitch), np.float32)
            zfull[:, :D] = z
            zb, bb = olm.reduce(ids, c["w"].astype(np.float32), lambda j: zfull[j], b32, 0, P)
            t, Mr, pr, Gs, v, new = olm.apply(th[o:o + pitch], M[:, o:o + pitch], p[o:o + pitch], zb, bb, k, alpha,
                                              float(sig[i]), 1.0, c, len(pidx), pidx, 0.001, 0.5)
            assert np.array_equal(eng.theta_cat.numpy()[o:o + pitch], t), (g, role)
            assert np.array_equal(eng.lmma_M.numpy()[:, o:o + pitch], Mr), (g, role)
            assert np.array_equal(eng.lmma_p.numpy()[o:o + pitch], pr), (g, role)
            assert np.array_equal(eng.lmma_G[i].numpy(), Gs), (g, role)
            assert eng.gstate[_lib.GS_SIGMA + i].item() == new == eng.history[g]["lmma"][role]["sigma_after"]
            assert eng.host_state()["sigma_history"][role][g + 1] == new      # recorded by the generation end


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(LM, record_history=False)
    full = _engine(4, **kw)
    for _ in range(5):
        full.step(sync=False)
    first = _engine(4, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "lm.pt")
    second = _engine(4, **kw)
    second.load_state_dict(torch.load(tmp_path / "lm.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    for name in ("gstate", "theta_cat", "lmma_M", "lmma_p", "lmma_G"):
        assert torch.equal(getattr(second, name), getattr(full, name)), name
    assert second.lmma_gen == full.lmma_gen == 5


def test_checkpoints_refuse_other_settings_and_parent_checkpoints_load():
    lm = _engine(4, record_history=False, **LM)
    lm.step(sync=False)
    sd = lm.state_dict()
    assert sd["es_distribution"] == {"es_distribution": "lmma", "sigma_learning_rate": None, "es_lmma_memory": 3}
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False, **dict(LM, es_lmma_memory=4)).load_state_dict(sd)
    # a checkpoint of the parent's code path: its es_distribution dict has no es_lmma_memory
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    old = plain.state_dict()
    old["es_distribution"] = {"es_distribution": "isotropic", "sigma_learning_rate": None}
    fresh = _engine(4, record_history=False)
    fresh.load_state_dict(old)
    assert torch.equal(fresh.theta_cat, plain.theta_cat) and torch.equal(fresh.gstate, plain.gstate)
    with pytest.raises(ValueError, match="distribution"):
        _engine(4, record_history=False, **LM).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    eng = _engine(P, comm=engine.Comm(), **LM)
    evs = [eng.step() for _ in range(3)]
    q.put(dict(rank=rank, evs=np.asarray(evs), rewards=np.stack([eng.history[g]["rewards"][r] for g in range(3)
                                                                 for r in ROLES]),
               theta=eng.theta_cat.numpy().copy(), M=eng.lmma_M.numpy().copy(), p=eng.lmma_p.numpy().copy(),
               G=eng.lmma_G.numpy().copy(), gstate=eng.gstate.numpy().copy()))
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
def test_lmma_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows; M, p, G and sigma are replicated."""
    single = _launch(1, 5, 29671)[0]
    two = _launch(2, 5, 29672)
    for o in two:
        assert np.array_equal(o["rewards"][:3], single["rewards"][:3])
        # the two ranks' partial recombinations are added in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], single["theta"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["M"], single["M"], rtol=0, atol=3e-5)
        np.testing.assert_allclose(o["p"], single["p"], rtol=0, atol=3e-5)
    for k in ("theta", "M", "p", "G", "gstate", "rewards"):
        assert np.array_equal(two[0][k], two[1][k]), k                 # replicas agree bit for bit
