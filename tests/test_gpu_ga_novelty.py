"""Co-GA novelty search on the GPU: the population + archive k-NN kernel bit for bit against the oracle on the
characterisation kernel's output for real members (with duplicates, row0 != 0, P = 1 and a P that needs several
candidate splits), the same bits for every split count and row block, the archive draw kernel bit for bit, the
wrappers' refusals, and the GA engine: w = 0 against the default, w = 1 and 0.5 against the oracle, determinism,
resume, the other GA options, and two GPUs."""
import os
import sys
import types

import numpy as np
import pytest
import torch

from oracle import es_novelty as en, es_options as oes, ga_es, ga_novelty as gn

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
SEED = 4242


def _n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _probe_obs(role, seed=SEED):
    from coevonet_b200 import ops
    states = ops.init_states(seed, en.PROBE_TAG, en.PROBES, "cuda")
    return ops.novelty_probe_obs(states, role)


def _bcs(P, role="agent_0", seed=SEED, sigma=0.05):
    """fp32 [P, 160] on the GPU: the characterisation kernel's output for P sigma-perturbed members."""
    from coevonet_b200 import layout, ops
    in_dim = layout.OBS_DIM[role]
    theta = ops.fc_init(in_dim, seed, role, 0, 1, "cuda")[0]
    rows = ops.es_perturb(theta, in_dim, sigma, seed, role, 0, 0, P)
    return ops.novelty_bc(rows, in_dim, _probe_obs(role, seed))


def _with_duplicates(pop, archive):
    """Copy some rows over others: equal members (zero distances, ties) and archive entries equal to members."""
    P = pop.shape[0]
    if P >= 4:
        pop[P - 1] = pop[0]
        pop[P // 2] = pop[1]
    if archive.shape[0] >= 2 and P >= 3:
        archive[0] = pop[2]
        archive[-1] = pop[P - 1]
    return pop, archive


# ---------------------------------------------------------------------------------------------------------------
# k-NN kernel
# ---------------------------------------------------------------------------------------------------------------
def _several_splits():
    return 2 * _n_sm() * 128 + 37


@pytest.mark.parametrize("P,n,row0,filled,k", [
    (1, 1, 0, 1, 1), (1, 1, 0, 7, 10), (1000, 1, 517, 0, 10), (1000, 300, 0, 64, 32), (1000, 300, 700, 1, 1),
    (1000, 300, 123, 1000, 10), ("several", 40, 12345, 100, 10)])
def test_knn_kernel_is_bit_exact(P, n, row0, filled, k):
    from coevonet_b200 import ops
    P = _several_splits() if P == "several" else P
    pop = _bcs(P)
    archive = _bcs(max(filled, 1), role="agent_1", seed=SEED + 1)[:filled].contiguous()
    pop, archive = _with_duplicates(pop, archive)
    ring = torch.zeros((max(filled, 1) + 3, 160), dtype=torch.float32, device="cuda")
    ring[:filled] = archive
    got = ops.ga_novelty_knn(pop[row0:row0 + n], row0, pop, ring, filled, k).cpu().numpy()
    want = gn.novelty(pop[row0:row0 + n].cpu().numpy(), row0, pop.cpu().numpy(), archive.cpu().numpy(), k)
    assert got.dtype == np.float64 and np.array_equal(got, want)
    assert np.all(np.isfinite(got))


def test_knn_kernel_duplicates_give_zero_and_id_exclusion():
    from coevonet_b200 import ops
    pop = _bcs(300)
    pop[17] = pop[5]
    ring = pop[40:41].clone()
    nov = ops.ga_novelty_knn(pop, 0, pop, ring, 1, 1).cpu().numpy()
    assert nov[5] == 0.0 and nov[17] == 0.0 and nov[40] == 0.0          # a copy elsewhere, never the member itself
    assert np.all(np.delete(nov, [5, 17, 40]) > 0.0)


def test_knn_kernel_nan_row():
    from coevonet_b200 import ops
    pop = _bcs(300)
    pop[9, 33] = float("nan")
    ring = _bcs(4, seed=SEED + 2)
    got = ops.ga_novelty_knn(pop, 0, pop, ring, 4, 10).cpu().numpy()
    want = gn.novelty(pop.cpu().numpy(), 0, pop.cpu().numpy(), ring.cpu().numpy(), 10)
    assert np.isnan(got[9]) and np.isnan(want[9])
    keep = np.arange(300) != 9
    assert np.array_equal(got[keep], want[keep]) and np.all(np.isfinite(got[keep]))


def test_knn_splits_and_row_blocks_give_identical_bits():
    """Split counts 1, the automatic count and one beyond the candidate tiles; and a population sharded into
    uneven row blocks gives the bits of one call over all rows."""
    from coevonet_b200 import ops
    P = _several_splits()
    pop = _bcs(P)
    ring = _bcs(1024, seed=SEED + 3)
    pop, ring = _with_duplicates(pop, ring)
    ref = ops.ga_novelty_knn(pop, 0, pop, ring, 1024, 10, splits=0)
    for s in (1, 3, 100000):
        assert torch.equal(ops.ga_novelty_knn(pop, 0, pop, ring, 1024, 10, splits=s), ref), s
    parts = []
    for a, b in ((0, 4000), (4000, 4001), (4001, P)):
        parts.append(ops.ga_novelty_knn(pop[a:b], a, pop, ring, 1024, 10))
    assert torch.equal(torch.cat(parts), ref)
    # the member block is read with its own row pitch: one role's column of a gathered [P, 3, 160] block
    block = torch.zeros((P, 3, 160), dtype=torch.float32, device="cuda")
    block[:, 1] = pop
    block[:, 0] = float("nan")
    assert torch.equal(ops.ga_novelty_knn(block[:, 1], 0, block[:, 1], ring, 1024, 10), ref)
    # deterministic
    assert torch.equal(ops.ga_novelty_knn(pop, 0, pop, ring, 1024, 10), ref)


def test_knn_wrapper_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    pop = _bcs(8)
    ring = torch.zeros((4, 160), dtype=torch.float32, device="cuda")
    bad = [
        lambda: ops.ga_novelty_knn(pop.cpu(), 0, pop.cpu(), ring.cpu(), 1, 3),                      # CPU
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, 1, 0),                                        # k
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, 1, 33),
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, 5, 3),                                        # filled > A
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, -1, 3),
        lambda: ops.ga_novelty_knn(pop[:1], 0, pop[:1], ring, 0, 3),                                # no candidate
        lambda: ops.ga_novelty_knn(pop, 1, pop, ring, 1, 3),                                        # rows past P
        lambda: ops.ga_novelty_knn(pop[:4], 5, pop, ring, 1, 3),
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, 1, 3, splits=-1),
        lambda: ops.ga_novelty_knn(pop.double(), 0, pop, ring, 1, 3),                               # dtype
        lambda: ops.ga_novelty_knn(pop[:, :128], 0, pop, ring, 1, 3),                               # width
        lambda: ops.ga_novelty_knn(pop, 0, pop.t().contiguous().t(), ring, 1, 3),                   # columns
        lambda: ops.ga_novelty_knn(pop, 0, torch.zeros((8, 161), device="cuda")[:, 1:], ring, 1, 3),  # alignment
        lambda: ops.ga_novelty_knn(pop, 0, pop, ring, 1, 3, out=torch.empty(8, device="cuda")),    # out dtype
    ]
    for i, fn in enumerate(bad):
        with pytest.raises(_lib.CevError):
            fn()
            pytest.fail(f"case {i} was accepted")
    # empty member block: nothing to do
    assert ops.ga_novelty_knn(pop[:0], 0, pop, ring, 1, 3).shape == (0,)


# ---------------------------------------------------------------------------------------------------------------
# archive draws
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("m,P", [(1, 1), (1, 7), (37, 1000), (4096, 65536), (300, 1 << 32)])
def test_draw_kernel_is_bit_exact(m, P):
    from coevonet_b200 import ops
    for gen in (0, 5, 123456):
        for role in ROLES:
            got = ops.ga_novelty_draw(SEED, gen, role, m, P, "cuda").cpu().numpy()
            assert np.array_equal(got, gn.draw_ids(SEED, gen, role, m, P)), (gen, role)


def test_draw_wrapper_refuses_bad_arguments():
    from coevonet_b200 import _lib, ops
    for fn in (lambda: ops.ga_novelty_draw(1, 0, "agent_0", 4, 0, "cuda"),
               lambda: ops.ga_novelty_draw(1, 0, "agent_0", 4, (1 << 32) + 1, "cuda"),
               lambda: ops.ga_novelty_draw(1, 0, "agent_0", 4, 8, "cpu"),
               lambda: ops.ga_novelty_draw(1, 0, "agent_0", 4, 8, "cuda", out=torch.empty(4, device="cuda"))):
        with pytest.raises(_lib.CevError):
            fn()


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


NOV = dict(ga_novelty_weight=0.5, ga_novelty_k=4, ga_novelty_archive=5, ga_novelty_archive_add=2)


def _bits(eng):
    eng.check_status()
    out = {"gstate": eng.gstate.cpu().numpy()}
    for r in ROLES:
        out["pop_" + r] = eng.pop[r].cpu().numpy().view(np.uint32)
        out["hof_" + r] = eng.hof[r].cpu().numpy().view(np.uint32)
        out["fit_" + r] = eng.fitness[r].cpu().numpy()
        out["elite_" + r] = eng.elite_ids[r].cpu().numpy()
        if eng.novelty_w:
            out["nov_" + r] = eng.novelty[r].cpu().numpy()
            out["F_" + r] = eng.shaped_fitness[r].cpu().numpy()
    if eng.novelty_ring is not None:
        out["ring"] = eng.novelty_ring.cpu().numpy().view(np.uint32)
    return out


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_zero_weight_equals_the_default_engine():
    plain = _engine(64)
    off = _engine(64, ga_novelty_weight=0.0)
    for _ in range(3):
        plain.step(sync=False)
        off.step(sync=False)
        _same(_bits(plain), _bits(off))
    assert off.novelty_ring is None


@pytest.mark.parametrize("w", [1.0, 0.5], ids=["novelty", "equal"])
def test_generations_match_the_oracle(w):
    """P = 48, A = 5, m = 2 over 4 generations (the ring wraps): the novelty is the oracle's k-NN of the kernel's
    characterisations of the evaluated members against the others and the ring as it stood; F, the elites, the
    fitness-best Hall-of-Fame row, the drawn ids and the rings follow the oracle."""
    from coevonet_b200 import layout, ops
    P, A, k, m, E = 48, 5, 4, 2, 4
    eng = _engine(P, record_history=True, ga_novelty_weight=w, ga_novelty_k=k, ga_novelty_archive=A,
                  ga_novelty_archive_add=m)
    obs = {r: _probe_obs(r) for r in ROLES}
    for i, r in enumerate(ROLES):
        assert torch.equal(eng.novelty_probe_obs[r], obs[r])
        assert torch.equal(eng.novelty_ring[i, 0], ops.novelty_bc(eng.founder[r].reshape(1, -1), layout.OBS_DIM[r],
                                                                  obs[r])[0])
    for g in range(4):
        before = {r: eng.pop[r].clone() for r in ROLES}
        ring = eng.novelty_ring.cpu().numpy().copy()
        filled, head = eng.novelty_filled, eng.novelty_head
        eng.step()
        h = eng.history[g]
        assert h["novelty_filled"] == filled
        for i, r in enumerate(ROLES):
            bcs = ops.novelty_bc(before[r], layout.OBS_DIM[r], obs[r]).cpu().numpy()
            N = gn.novelty(bcs, 0, bcs, ring[i, :filled], k)
            assert np.array_equal(h["novelty"][r], N), (g, r)
            R = h["fitness"][r]
            F = en.combine(oes.centered_ranks(R), oes.centered_ranks(N), w)
            assert np.array_equal(h["shaped_fitness"][r], F), (g, r)
            ids = ga_es.select_topk(F, E, 1)
            assert np.array_equal(h["elite_ids"][r], ids), (g, r)
            best = ga_es.select_topk(R, 1, 1)[0]
            assert torch.equal(eng.hof[r][-1], before[r][best]), (g, r)
            assert torch.equal(eng.pop[r][0], before[r][ids[0]]), (g, r)
            drawn = gn.draw_ids(SEED, g, r, m, P)
            assert np.array_equal(h["novelty_archive_ids"][r], drawn), (g, r)
            for j, d in enumerate(drawn):
                ring[i, (head + j) % A] = bcs[d]
            assert np.array_equal(eng.novelty_ring[i].cpu().numpy(), ring[i]), (g, r)
        assert eng.novelty_filled == min(filled + m, A)
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


@pytest.mark.parametrize("opts", [dict(crossover_rate=0.3), dict(adaptive=True), dict(fitness_sharing=False),
                                  dict(reference_compat=False, fitness_sharing=True),
                                  dict(play_discarded_hof_games=True)],
                         ids=["crossover", "adaptive", "no_sharing", "no_reference_compat", "discarded_hof_games"])
def test_composes_with_the_other_options(opts):
    eng = _engine(64, record_history=True, **dict(NOV, **opts))
    for g in range(2):
        eng.step()
        h = eng.history[g]
        for r in ROLES:
            N, R, F = h["novelty"][r], h["fitness"][r], h["shaped_fitness"][r]
            assert np.all(np.isfinite(N)) and np.all(N > 0)
            assert np.array_equal(F, en.combine(oes.centered_ranks(R), oes.centered_ranks(N), 0.5))
            assert np.array_equal(h["elite_ids"][r], ga_es.select_topk(F, 4, eng.order))
    eng.check_status()
    assert all(np.all(np.isfinite(eng.pop[r].cpu().numpy())) for r in ROLES)


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
    args = _args(P, record_history=True, **NOV)
    pop, hof, founder = _rows(P, int(args.hof_size), dev, shard.row0, shard.n_local)
    eng = engine.GAEngine(args, dev, pop, hof, founder, comm=comm)
    for _ in range(3):
        eng.step()
    rec = {key: np.stack([eng.history[g][key][r] for g in range(3) for r in ROLES])
           for key in ("fitness", "novelty", "shaped_fitness", "elite_ids", "novelty_archive_ids")}
    q.put((rank, dict(ring=eng.novelty_ring.cpu().numpy(), row0=shard.row0, n_local=shard.n_local,
                      hof=np.concatenate([eng.hof[r].cpu().numpy() for r in ROLES], axis=1),
                      pop=np.concatenate([eng.pop[r].cpu().numpy() for r in ROLES], axis=1), **rec)))
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
def test_novelty_sharded_over_two_gpus_equal_one_gpu():
    P = 387                                        # 194 + 193 rows
    one = _launch(1, P, 29751)[0]
    two = _launch(2, P, 29752)
    for o in two:
        for key in ("novelty", "shaped_fitness", "elite_ids", "novelty_archive_ids", "ring", "hof"):
            assert np.array_equal(o[key], one[key]), key
        np.testing.assert_allclose(o["fitness"], one["fitness"], rtol=1e-12, atol=0)
        assert np.array_equal(o["pop"], one["pop"][o["row0"]:o["row0"] + o["n_local"]])
