"""Co-ES LM-MA-ES on the GPU: the projection, the LM-MA K5, the recombination and the apply against oracle/es_lmma.py
bit for bit given the kernels' own normals (the K5 stream; libm and MUFU normals differ in the last bits), the
projection's independence of row blocks and grids, the status word, and the engine against the oracle generation by
generation, determinism, resume and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_lmma as olm

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 4242


def _noise(theta, in_dim, role, gen, row0, n):
    """The kernel's normals of members [row0, row0 + n): fp32 [n, pitch], zero off the Linear entries."""
    from coevonet_b200 import ops
    noise = torch.empty((n, theta.numel()), device="cuda")
    sig = torch.tensor([0.01], dtype=torch.float64, device="cuda")
    ops.es_perturb(theta, in_dim, sig, SEED, role, gen, row0, n, noise_out=noise)
    return noise


def _vectors(in_dim, m, seed, scale=1.0, collinear=False):
    from coevonet_b200 import layout
    from oracle import layout as olayout
    rng = np.random.default_rng(seed)
    M = np.zeros((m, layout.fc_pitch(in_dim)), np.float32)
    pidx = olayout.fc_perturbable_index(in_dim)
    M[:, pidx] = rng.standard_normal((m, len(pidx))) * scale
    if collinear and m > 1:
        M[1, pidx] = M[0, pidx] * np.float32(1 + 1e-6)
    return M


def _gram(M):
    M64 = M.astype(np.float64)
    return M64 @ M64.T


@pytest.mark.parametrize("role,k,m", [("agent_0", 1, 8), ("adversary_0", 5, 8), ("agent_1", 16, 16),
                                      ("agent_0", 32, 32)])
def test_projection_and_coefficients_match_the_oracle_bit_for_bit(role, k, m):
    from coevonet_b200 import engine, layout, ops
    in_dim = layout.OBS_DIM[role]
    D = layout.fc_dim(in_dim)
    theta = ops.fc_init(in_dim, 5, role, 0, 1, "cuda")[0]
    M = _vectors(in_dim, m, 3, collinear=True)
    G = _gram(M)
    c = engine.lmma_constants(1024, D, m)
    row0, n = 13, 70
    Md, Gd = torch.from_numpy(M).cuda(), torch.from_numpy(G).cuda()
    s_out = torch.empty((n, k), dtype=torch.float64, device="cuda")
    beta = ops.es_lmma_project(Md, k, Gd, c["c_d"][:k], in_dim, SEED, role, 2, row0, n, s_out=s_out)
    z = _noise(theta, in_dim, role, 2, row0, n).cpu().numpy()[:, :D]
    s = olm.project(M[:, :D], z, k)
    assert np.array_equal(s_out.cpu().numpy(), s)
    _, b = olm.transform_compact(s, G, k, c["c_d"])
    assert np.array_equal(beta.cpu().numpy(), b.astype(np.float32))
    # K5 given the device's beta, bit for bit
    from oracle import layout as olayout
    sig = torch.tensor([0.03], dtype=torch.float64, device="cuda")
    rows = ops.es_perturb_lmma(theta, in_dim, sig, Md, k, beta, c["alpha"][k], SEED, role, 2, row0, n)
    want = olm.perturb(theta.cpu().numpy()[:D], np.float32(0.03), M[:, :D], beta.cpu().numpy(), c["alpha"][k], z,
                       olayout.fc_perturbable_index(in_dim))
    got = rows.cpu().numpy()
    assert np.array_equal(got[:, :D], want) and not np.any(got[:, D:])


def test_projection_bits_do_not_depend_on_row_blocks_shards_or_grid():
    from coevonet_b200 import engine, layout, ops
    role, k, m = "agent_1", 8, 8
    in_dim = layout.OBS_DIM[role]
    M = torch.from_numpy(_vectors(in_dim, m, 7)).cuda()
    G = torch.from_numpy(_gram(M.cpu().numpy())).cuda()
    cd = engine.lmma_constants(512, layout.fc_dim(in_dim), m)["c_d"]
    full = ops.es_lmma_project(M, k, G, cd, in_dim, SEED, role, 4, 0, 300)
    for cuts in ((0, 1, 300), (0, 64, 65, 300), (0, 137, 300), (0, 299, 300)):
        parts = [ops.es_lmma_project(M, k, G, cd, in_dim, SEED, role, 4, a, b - a) for a, b in zip(cuts, cuts[1:])]
        assert torch.equal(torch.cat(parts), full), cuts


def test_k5_with_zero_beta_is_the_isotropic_k5():
    from coevonet_b200 import layout, ops
    role = "adversary_0"
    in_dim = layout.OBS_DIM[role]
    theta = ops.fc_init(in_dim, 5, role, 0, 1, "cuda")[0]
    sig = torch.tensor([0.05], dtype=torch.float64, device="cuda")
    M = torch.from_numpy(_vectors(in_dim, 4, 2)).cuda()
    for row0, n in ((0, 64), (7, 41)):
        beta = torch.zeros((n, 4), device="cuda")
        got = ops.es_perturb_lmma(theta, in_dim, sig, M, 4, beta, 1.0, SEED, role, 2, row0, n)
        assert torch.equal(got, ops.es_perturb(theta, in_dim, sig, SEED, role, 2, row0, n))


def _apply_inputs(m, k, seed, p_scale=1.0):
    from coevonet_b200 import layout, ops
    rng = np.random.default_rng(seed)
    dims = [layout.OBS_DIM[r] for r in ROLES]
    n = sum(layout.fc_pitch(d) for d in dims)
    theta = torch.cat([ops.fc_init(d, 5, r, 0, 1, "cuda")[0] for d, r in zip(dims, ROLES)])
    M = np.concatenate([_vectors(d, m, seed + i) for i, d in enumerate(dims)], axis=1)
    p = np.concatenate([_vectors(d, 1, seed + 10 + i, p_scale)[0] for i, d in enumerate(dims)])
    zbar = np.concatenate([_vectors(d, 1, seed + 20 + i, 0.05)[0] for i, d in enumerate(dims)])
    betabar = (rng.standard_normal((3, m)) * 1e-3).astype(np.float32)
    return dims, n, theta, M, p, zbar, betabar


@pytest.mark.parametrize("m,k,p_scale,bound", [(8, 3, 1.0, None), (4, 4, 30.0, "max"), (32, 17, 0.0, "min")])
def test_apply_gram_and_csa_match_the_oracle(m, k, p_scale, bound):
    from coevonet_b200 import _lib, engine, layout, ops
    from oracle import layout as olayout
    dims, n, theta, M, p, zbar, betabar = _apply_inputs(m, k, 11, p_scale)
    P = 256
    cs = [engine.lmma_constants(P, len(olayout.fc_perturbable_index(d)), m) for d in dims]
    gstate = ops.generation_state({None: [0.05, 0.2, 0.01], "max": [0.2, 0.3, 0.4], "min": [0.001] * 3}[bound], 16,
                                  "cuda")
    sig0 = gstate[_lib.GS_SIGMA:_lib.GS_SIGMA + 3].cpu().numpy().copy()
    th, Md, pd = theta.clone(), torch.from_numpy(M).cuda(), torch.from_numpy(p).cuda()
    G = torch.zeros((3, m, m), dtype=torch.float64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    smin, smax = 0.001, 0.5
    stats = ops.es_lmma_apply(th, Md, pd, torch.from_numpy(zbar).cuda(), torch.from_numpy(betabar).cuda(), dims, k=k,
                              alpha=[c["alpha"][k] for c in cs], c_sigma=[c["c_sigma"] for c in cs],
                              mu_w=[c["mu_w"] for c in cs], c_m=1.0, c_c=[c["c_c"] for c in cs], G=G, gstate=gstate,
                              sigma_min=smin, sigma_max=smax, status=status)
    assert status.item() == 0
    start = 0
    for s, d in enumerate(dims):
        sl = slice(start, start + layout.fc_pitch(d))
        pidx = olayout.fc_perturbable_index(d)
        t, Mr, pr, Gs, v, new = olm.apply(theta.cpu().numpy()[sl], M[:, sl], p[sl], zbar[sl], betabar[s], k,
                                          cs[s]["alpha"][k], float(sig0[s]), 1.0, cs[s], len(pidx), pidx, smin, smax)
        assert np.array_equal(th.cpu().numpy()[sl], t)
        assert np.array_equal(Md.cpu().numpy()[:, sl], Mr)
        assert np.array_equal(pd.cpu().numpy()[sl], pr)
        assert np.array_equal(G[s].cpu().numpy(), Gs)
        assert stats[s, 0].item() == v
        # exp of the device and of libm may differ in the last bit
        np.testing.assert_allclose(stats[s, 1].item(), new, rtol=1e-15)
        assert gstate[_lib.GS_SIGMA + s].item() == stats[s, 1].item()
        if bound == "max":
            assert new == smax
        if bound == "min":
            assert new == smin
        start = sl.stop


def test_reduction_matches_the_oracle_over_a_shard_boundary():
    from coevonet_b200 import engine, layout, ops
    role, P, k = "agent_0", 100, 3
    in_dim = layout.OBS_DIM[role]
    theta = ops.fc_init(in_dim, 5, role, 0, 1, "cuda")[0]
    c = engine.lmma_constants(P, layout.fc_dim(in_dim), k)
    rng = np.random.default_rng(5)
    fit = rng.standard_normal(P)
    ids = torch.from_numpy(np.argsort(-fit, kind="stable")[:c["mu"]].copy()).cuda()
    w = torch.tensor(c["w"], dtype=torch.float32).cuda()
    beta_all = (rng.standard_normal((P, k)) * 1e-2).astype(np.float32)
    z_all = _noise(theta, in_dim, role, 6, 0, P).cpu().numpy()
    total = np.zeros(layout.fc_pitch(in_dim))
    for row0, n in ((0, 37), (37, 63)):
        beta = torch.from_numpy(beta_all[row0:row0 + n].copy()).cuda()
        zb, bb = ops.es_lmma_reduce(ids, w, beta, in_dim, SEED, role, 6, row0, n)
        wz, wb = olm.reduce(ids.cpu().numpy(), w.cpu().numpy(), lambda i: z_all[i], beta_all[row0:row0 + n], row0, n)
        assert np.array_equal(zb.cpu().numpy(), wz) and np.array_equal(bb.cpu().numpy(), wb)
        total += zb.cpu().numpy()
    want = (c["w"].astype(np.float32).astype(np.float64) @ z_all[ids.cpu().numpy()].astype(np.float64))
    np.testing.assert_allclose(total, want, rtol=0, atol=1e-6)


def test_non_finite_inputs_set_the_status_word():
    from coevonet_b200 import engine, layout, ops
    role = "agent_0"
    in_dim = layout.OBS_DIM[role]
    M = _vectors(in_dim, 4, 1)
    M[2, 5] = np.inf
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    G = torch.from_numpy(_gram(np.nan_to_num(M))).cuda()
    cd = engine.lmma_constants(64, layout.fc_dim(in_dim), 4)["c_d"]
    ops.es_lmma_project(torch.from_numpy(M).cuda(), 4, G, cd, in_dim, SEED, role, 0, 0, 8, status=status)
    assert status.item() & 1
    dims, n, theta, M, p, zbar, betabar = _apply_inputs(4, 2, 3)
    p[7] = np.nan
    status.zero_()
    gstate = ops.generation_state([0.05, 0.05, 0.05], 16, "cuda")
    ops.es_lmma_apply(theta, torch.from_numpy(M).cuda(), torch.from_numpy(p).cuda(), torch.from_numpy(zbar).cuda(),
                      torch.from_numpy(betabar).cuda(), dims, k=2, alpha=[1.0] * 3, c_sigma=[0.01] * 3, mu_w=[2.0] * 3,
                      c_m=1.0, c_c=[[0.01] * 4] * 3, G=torch.zeros((3, 4, 4), dtype=torch.float64, device="cuda"),
                      gstate=gstate, sigma_min=0.001, sigma_max=0.5, status=status)
    assert status.item() & 1


# ---------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------
def _args(P, E=4, **opts):
    a = types.SimpleNamespace(
        algorithm="ES", generations=8, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.04, mutation_power_adversary=0.03,
        learning_rate=1.0, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=E, reference_compat=True, init_states="device", seed=SEED, plots=False,
        record_history=False, es_distribution="lmma", es_lmma_memory=3)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _engine(P, dev=None, comm=None, **opts):
    from coevonet_b200 import engine, layout, ops
    dev = dev or torch.device("cuda", 0)
    theta = {r: ops.fc_init(layout.OBS_DIM[r], 5, r, 0, 1, dev)[0].cpu() for r in ROLES}
    return engine.ESEngine(_args(P, **opts), dev, theta, comm=comm)


def _bits(eng):
    eng.check_status()
    out = {"theta": eng.theta_cat.cpu().numpy().view(np.uint32), "gstate": eng.gstate.cpu().numpy(),
           "M": eng.lmma_M.cpu().numpy().view(np.uint32), "p": eng.lmma_p.cpu().numpy().view(np.uint32),
           "G": eng.lmma_G.cpu().numpy()}
    for r in ROLES:
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
    return out


def test_engine_follows_the_oracle_generation_by_generation():
    """Three generations with the Hall of Fame (k = 0, 1, 2): the members against the oracle's K5 given the oracle's
    projection of the kernel's normals, then theta, M, p, G and sigma against the oracle's recombination and apply
    on the engine's fitness."""
    from coevonet_b200 import _lib, layout
    from oracle import layout as olayout
    P = 64
    eng = _engine(P, es_hof_size=3, es_hof_opponents=2)
    for g in range(3):
        th, M, p = (x.cpu().numpy().copy() for x in (eng.theta_cat, eng.lmma_M, eng.lmma_p))
        G = eng.lmma_G.cpu().numpy().copy()
        sig = eng.gstate[_lib.GS_SIGMA:_lib.GS_SIGMA + 3].cpu().numpy().copy()
        k = min(g, 3)
        eng.step(sync=False)
        eng.check_status()
        for i, role in enumerate(ROLES):
            o, pitch = eng.cols[role]
            in_dim = layout.OBS_DIM[role]
            D = layout.fc_dim(in_dim)
            pidx = olayout.fc_perturbable_index(in_dim)
            c = eng.lmma_const[role]
            z = _noise(eng.theta[role], in_dim, role, g, 0, P).cpu().numpy()
            s = olm.project(M[:, o:o + D], z[:, :D], k) if k else np.zeros((P, 0))
            _, b = olm.transform_compact(s, G[i], k, c["c_d"])
            b32 = b.astype(np.float32)
            rows = olm.perturb(th[o:o + D], np.float32(sig[i]), M[:, o:o + D], b32, c["alpha"][k], z[:, :D], pidx)
            assert np.array_equal(eng.members[role].cpu().numpy()[:, :D], rows), (g, role)
            fit = eng.fitness[role].cpu().numpy()
            ids = np.argsort(-fit, kind="stable")[:c["mu"]]
            zb, bb = olm.reduce(ids, c["w"].astype(np.float32), lambda j: z[j], b32, 0, P)
            t, Mr, pr, Gs, v, new = olm.apply(th[o:o + pitch], M[:, o:o + pitch], p[o:o + pitch], zb, bb, k,
                                              c["alpha"][k], float(sig[i]), 1.0, c, len(pidx), pidx, 0.001, 0.5)
            assert np.array_equal(eng.theta_cat.cpu().numpy()[o:o + pitch], t), (g, role)
            assert np.array_equal(eng.lmma_M.cpu().numpy()[:, o:o + pitch], Mr), (g, role)
            assert np.array_equal(eng.lmma_p.cpu().numpy()[o:o + pitch], pr), (g, role)
            assert np.array_equal(eng.lmma_G[i].cpu().numpy(), Gs), (g, role)
            np.testing.assert_allclose(eng.gstate[_lib.GS_SIGMA + i].item(), new, rtol=1e-15)


def test_lmma_engine_deterministic_and_resume_bit_exact(tmp_path):
    kw = dict(es_hof_size=2, es_hof_opponents=2, es_lmma_memory=4)
    runs = []
    for _ in range(2):
        eng = _engine(64, **kw)
        for _ in range(5):
            eng.step(sync=False)
        runs.append(_bits(eng))
    for key in runs[0]:
        assert np.array_equal(runs[0][key], runs[1][key]), key
    first = _engine(64, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "lmma.pt")
    second = _engine(64, **kw)
    second.load_state_dict(torch.load(tmp_path / "lmma.pt", weights_only=False))
    for _ in range(3):
        second.step(sync=False)
    res = _bits(second)
    for key in runs[0]:
        assert np.array_equal(runs[0][key], res[key]), key


def _worker(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from coevonet_b200 import engine
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    eng = _engine(P, dev=dev, comm=engine.Comm())
    for _ in range(3):
        eng.step(sync=False)
    q.put((rank, dict(theta=eng.theta_cat.cpu().numpy(), M=eng.lmma_M.cpu().numpy(), p=eng.lmma_p.cpu().numpy(),
                      G=eng.lmma_G.cpu().numpy(), gstate=eng.gstate.cpu().numpy())))
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
def test_lmma_sharded_over_two_gpus_equal_one_gpu():
    P = 193                                        # 97 + 96 rows
    one = _launch(1, P, 29751)[0]
    two = _launch(2, P, 29752)
    for k in two[0]:
        assert np.array_equal(two[0][k], two[1][k]), k             # replicas agree bit for bit
    for o in two:
        # the all-reduce adds the ranks' partial recombinations in another order: fp32 rounding only
        np.testing.assert_allclose(o["theta"], one["theta"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(o["M"], one["M"], rtol=0, atol=1e-5)
        np.testing.assert_allclose(o["p"], one["p"], rtol=0, atol=1e-5)
