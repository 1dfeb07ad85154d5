"""Co-GA novelty search on the host: the oracle's fmaf emulation against exact rounding, its population + archive k-NN
against a brute-force restatement, the archive draws, flag validation, and the GA engine's novelty path with the
checker backend (tests/ga_novelty_backend.py): the default call log at w = 0, the selection fitness, elites, Hall of
Fame rows and archive rings against the oracle over several generations, resume, checkpoints and two gloo ranks."""
import os
import sys
import types
from fractions import Fraction

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import es_novelty as en, es_options as oes, ga_es, ga_novelty as gn, philox

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLES = ("agent_0", "agent_1", "adversary_0")
NOV = dict(ga_novelty_weight=0.5, ga_novelty_k=3, ga_novelty_archive=4, ga_novelty_archive_add=2)


# ---------------------------------------------------------------------------------------------------------------
# the oracle
# ---------------------------------------------------------------------------------------------------------------
def _round32(x):
    """Exact rational -> nearest float32, ties to even."""
    r = np.float32(float(x))
    cands = (np.nextafter(r, np.float32(-np.inf)), r, np.nextafter(r, np.float32(np.inf)))
    return min(cands, key=lambda y: (abs(Fraction(float(y)) - x), int(np.array(y).view(np.uint32)) & 1))


def test_fma32_emulation_against_exact_rounding():
    rng = np.random.default_rng(0)
    a = rng.normal(size=50000).astype(np.float32)
    b = rng.normal(size=50000).astype(np.float32)
    c = rng.normal(size=50000).astype(np.float32)
    got = gn.fma32(a, b, c)
    for i in range(0, 50000, 499):
        assert got[i] == _round32(Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i])))
    # the distance's own form: squares added to a non-negative running sum of another magnitude
    e = (rng.random(20000) * 2.0 ** rng.integers(-20, 4, 20000)).astype(np.float32)
    s = (rng.random(20000) * 2.0 ** rng.integers(-10, 8, 20000)).astype(np.float32)
    got = gn.fma32(e, e, s)
    for i in range(0, 20000, 199):
        assert got[i] == _round32(Fraction(float(e[i])) ** 2 + Fraction(float(s[i])))
    # exactly 2^-70 below a float32 midpoint, where the fp64 sum lands: a second rounding would go up
    c1 = np.array([np.float32(1 + 2.0 ** -23)])
    x = gn.fma32(np.array([np.float32(2.0 ** -24 * (1 - 2.0 ** -23))]), np.array([np.float32(1 + 2.0 ** -23)]), c1)
    assert (c1.astype(np.float64) + 2.0 ** -24 * (1 - 2.0 ** -46)).astype(np.float32)[0] != c1[0]
    assert x[0] == c1[0]


def _brute_dist(q, x):
    """One pair, one operation at a time: fl32(q_t - x_t), the fmaf rounded exactly, the fp32 square root."""
    s = np.float32(0.0)
    for t in range(len(q)):
        e = np.float32(q[t]) - np.float32(x[t])
        if not (np.isfinite(e) and np.isfinite(s)):
            s = np.float32(np.nan) if (np.isnan(e) or np.isnan(s)) else np.float32(np.inf)
            continue
        s = _round32(Fraction(float(e)) ** 2 + Fraction(float(s)))
    return np.float32(np.sqrt(s))


def _brute_novelty(x, row0, pop, archive, k):
    cands = list(pop) + list(archive)
    out = []
    for i, q in enumerate(x):
        pairs = []
        for c, y in enumerate(cands):
            if c == row0 + i:
                continue
            d = _brute_dist(q, y)
            pairs.append(((1, 0.0, c) if np.isnan(d) else (0, float(d), c), d))
        ke = min(k, len(pop) - 1 + len(archive))
        acc = 0.0
        for _, d in sorted(pairs, key=lambda p: p[0])[:ke]:
            acc += float(d)
        out.append(acc / ke)
    return np.array(out)


def _bcs(rng, n):
    return rng.dirichlet(np.ones(5), size=(n, 32)).reshape(n, 160).astype(np.float32)


@pytest.mark.parametrize("P,filled,row0,n,k", [(6, 3, 0, 6, 2), (6, 3, 2, 3, 4), (5, 0, 0, 5, 10), (1, 3, 0, 1, 2),
                                               (1, 1, 0, 1, 32), (7, 5, 4, 3, 32)])
def test_knn_equals_brute_force(P, filled, row0, n, k):
    rng = np.random.default_rng(P * 100 + filled * 10 + k)
    pop = _bcs(rng, P)
    archive = _bcs(rng, filled)
    x = pop[row0:row0 + n]
    got = gn.novelty(x, row0, pop, archive, k)
    assert got.dtype == np.float64
    want = _brute_novelty(x, row0, pop, archive, k)
    assert np.array_equal(got, want)


def test_knn_self_exclusion_duplicates_and_nan():
    rng = np.random.default_rng(7)
    base = _bcs(rng, 3)
    # rows 0 and 1 are duplicates (zero distances, ties broken by index), row 3 duplicates the archive entry
    pop = np.concatenate([base[:1], base[:1], base[1:3], _bcs(rng, 2)])
    archive = np.concatenate([pop[3:4], _bcs(rng, 1)])
    for k in (1, 2, 3, 7, 32):
        got = gn.novelty(pop, 0, pop, archive, k)
        assert np.array_equal(got, _brute_novelty(pop, 0, pop, archive, k)), k
    # excluded by id, not by value: row 0's nearest is its duplicate row 1 at distance 0
    assert gn.novelty(pop[:1], 0, pop, archive, 1)[0] == 0.0
    assert gn.novelty(pop[3:4], 3, pop, archive, 1)[0] == 0.0                # the archive's copy of itself
    assert gn.novelty(pop[2:3], 2, pop, archive, 1)[0] > 0.0
    # a NaN row: its own distances are all NaN, so its novelty is NaN; the others sort it last and never reach it
    bad = pop.copy()
    bad[4, 17] = np.nan
    got = gn.novelty(bad, 0, bad, archive, 32)
    want = _brute_novelty(bad, 0, bad, archive, 32)
    assert np.isnan(got[4]) and np.isnan(want[4])
    assert all(np.isnan(got[i]) for i in range(len(bad)))                       # k_eff = 7 reaches the NaN one
    got = gn.novelty(bad, 0, bad, archive, 3)
    want = _brute_novelty(bad, 0, bad, archive, 3)
    keep = np.arange(len(bad)) != 4
    assert np.array_equal(got[keep], want[keep]) and np.isnan(got[4])
    # the NaN candidate sorts after +inf
    d = np.array([np.nan, np.inf, 1.0], np.float32)
    assert list(np.argsort(gn.sort_keys(d, np.arange(3)))) == [2, 1, 0]


def test_knn_needs_a_candidate():
    with pytest.raises(ValueError):
        gn.novelty(_bcs(np.random.default_rng(1), 1), 0, _bcs(np.random.default_rng(1), 1), np.zeros((0, 160)), 3)


def test_draw_ranges_and_keying():
    for P in (1, 2, 7, 65536, 1 << 32):
        ids = gn.draw_ids(99, 3, "agent_1", 37, P)
        assert ids.dtype == np.int64 and ids.shape == (37,)
        assert ids.min() >= 0 and ids.max() < P
    assert not np.any(gn.draw_ids(99, 3, "agent_1", 37, 1))
    # the multiply-shift of word (j & 3) of Philox block j >> 2 at (member 0, gen, role | kind << 8)
    w = philox.words(99, 9, 1, 3, [0], 10).reshape(-1)
    want = [(int(w[j]) * 1000) >> 32 for j in range(37)]
    assert gn.draw_ids(99, 3, "agent_1", 37, 1000).tolist() == want
    # a prefix of a longer draw; other generations, roles, seeds draw other ids
    assert np.array_equal(gn.draw_ids(99, 3, 1, 5, 1000), gn.draw_ids(99, 3, 1, 37, 1000)[:5])
    base = gn.draw_ids(99, 3, 1, 16, 1 << 20)
    for other in (gn.draw_ids(99, 4, 1, 16, 1 << 20), gn.draw_ids(99, 3, 2, 16, 1 << 20),
                  gn.draw_ids(98, 3, 1, 16, 1 << 20)):
        assert not np.array_equal(base, other)


# ---------------------------------------------------------------------------------------------------------------
# flags
# ---------------------------------------------------------------------------------------------------------------
def _cli(argv):
    from coevonet_b200.main import Args, parse_arguments
    return Args(parse_arguments(argv))


def test_novelty_flags_defaults_and_parsing():
    from coevonet_b200.engine import GA_NOVELTY_DEFAULTS, ga_novelty as validate
    a = _cli(["--algorithm=GA"])
    assert (a.ga_novelty_weight, a.ga_novelty_k, a.ga_novelty_archive, a.ga_novelty_archive_add) == \
        (0.0, None, None, None)
    assert validate(a) == GA_NOVELTY_DEFAULTS
    assert validate(types.SimpleNamespace(algorithm="GA")) == GA_NOVELTY_DEFAULTS                # attributes absent
    assert validate(types.SimpleNamespace(population=4)) == GA_NOVELTY_DEFAULTS
    assert validate(_cli(["--algorithm=GA", "--ga_novelty_weight=1"])) == \
        {"ga_novelty_weight": 1.0, "ga_novelty_k": 10, "ga_novelty_archive": 1024, "ga_novelty_archive_add": 1}
    assert validate(_cli(["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_k=32", "--ga_novelty_archive=1",
                          "--ga_novelty_archive_add=1"])) == \
        {"ga_novelty_weight": 0.5, "ga_novelty_k": 32, "ga_novelty_archive": 1, "ga_novelty_archive_add": 1}
    assert validate(_cli(["--algorithm=GA", "--ga_novelty_weight=0.25", "--ga_novelty_k=1",
                          "--ga_novelty_archive=32768", "--ga_novelty_archive_add=32768"]))["ga_novelty_archive_add"] \
        == 32768
    assert validate(_cli(["--algorithm=ES", "--ga_novelty_weight=0"])) == GA_NOVELTY_DEFAULTS
    # the existing Co-ES refusals for the GA are unchanged, and the ES novelty flags still belong to the ES
    with pytest.raises(ValueError, match="GA"):
        _cli(["--algorithm=GA", "--es_novelty_weight=0.5", "--ga_novelty_weight=0.5"])


@pytest.mark.parametrize("argv,match", [
    (["--algorithm=ES", "--ga_novelty_weight=0.5"], "ES"),
    (["--algorithm=ES", "--ga_novelty_k=4"], "ES"),
    (["--algorithm=ES", "--ga_novelty_archive=4"], "ES"),
    (["--algorithm=ES", "--ga_novelty_archive_add=4"], "ES"),
    (["--algorithm=GA", "--ga_novelty_weight=1.5"], r"\[0, 1\]"),
    (["--algorithm=GA", "--ga_novelty_weight=-0.1"], r"\[0, 1\]"),
    (["--algorithm=GA", "--ga_novelty_weight=nan"], r"\[0, 1\]"),
    (["--algorithm=GA", "--ga_novelty_weight=inf"], r"\[0, 1\]"),
    (["--algorithm=GA", "--ga_novelty_k=4"], "needs ga_novelty_weight"),
    (["--algorithm=GA", "--ga_novelty_archive=64"], "needs ga_novelty_weight"),
    (["--algorithm=GA", "--ga_novelty_archive_add=2"], "needs ga_novelty_weight"),
    (["--algorithm=GA", "--ga_novelty_weight=0", "--ga_novelty_k=10"], "needs ga_novelty_weight"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_k=0"], r"\[1, 32\]"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_k=33"], r"\[1, 32\]"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_archive=0"], r"\[1, 32768\]"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_archive=32769"], r"\[1, 32768\]"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_archive_add=0"], r"\[1, ga_novelty_archive"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_archive_add=1025"], r"\[1, ga_novelty_archive"),
    (["--algorithm=GA", "--ga_novelty_weight=0.5", "--ga_novelty_archive=8", "--ga_novelty_archive_add=9"],
     r"\[1, ga_novelty_archive = 8\]"),
])
def test_novelty_refusals(argv, match):
    with pytest.raises(ValueError, match=match):
        _cli(["--population=8"] + argv)


def test_engines_refuse_bad_novelty_settings():
    from coevonet_b200 import engine
    with pytest.raises(ValueError, match="ES"):
        engine.ESEngine(_args(4, algorithm="ES", ga_novelty_weight=0.5), "cpu", {}, kernels=_backend())
    with pytest.raises(ValueError, match=r"\[0, 1\]"):
        _engine(4, ga_novelty_weight=2.0)
    with pytest.raises(ValueError, match="GA"):
        _engine(4, es_novelty_weight=0.5)


# ---------------------------------------------------------------------------------------------------------------
# engine on the checker backend
# ---------------------------------------------------------------------------------------------------------------
def _backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ga_novelty_backend
    return ga_novelty_backend


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
        algorithm="GA", generations=8, population=P, hof_size=2, game="simple_adversary_v3",
        mutation_power_agent_0=0.05, mutation_power_agent_1=0.04, mutation_power_adversary=0.03,
        learning_rate=0.1, max_timesteps_per_episode=400, max_evaluation_steps=400, elites_number=2,
        adaptive=False, max_mutation_power=0.5, min_mutation_power=0.001, fitness_sharing=True,
        early_stopping=False, patience=300, min_delta=0.1, debug=False, precision="float32", save=False,
        envs_per_member=1, reference_compat=True, init_states="device", seed=99, plots=False,
        record_history=record_history)
    for k, v in opts.items():
        setattr(a, k, v)
    return a


def _rows(P, seed=700):
    from coevonet_b200 import layout
    from oracle import weights
    pop, hof, founder = {}, {}, {}
    for i, r in enumerate(ROLES):
        in_dim = layout.OBS_DIM[r]
        rows = np.zeros((P + 3, layout.fc_pitch(in_dim)), dtype=np.float32)
        rows[:, :layout.fc_dim(in_dim)] = weights.make_fc_rows(P + 3, in_dim, seed + i, ln_jitter=0.02)
        pop[r] = torch.from_numpy(rows[:P].copy())
        hof[r] = torch.from_numpy(rows[P:P + 2].copy())
        founder[r] = torch.from_numpy(rows[P + 2].copy())
    return pop, hof, founder


def _engine(P, comm=None, kernels=None, **kw):
    from coevonet_b200 import engine
    pop, hof, founder = _rows(P)
    shard = engine.Shard(P, comm.rank if comm else 0, comm.world if comm else 1)
    sl = slice(shard.row0, shard.row0 + shard.n_local)
    return engine.GAEngine(_args(P, **kw), "cpu", {r: pop[r][sl].clone() for r in ROLES}, hof, founder,
                           kernels=kernels or _backend(), comm=comm)


def test_zero_weight_issues_the_default_calls():
    logs, states = [], []
    for kw in ({}, {"ga_novelty_weight": 0.0}):
        log = _Log()
        eng = _engine(4, kernels=log, **kw)
        for _ in range(2):
            eng.step()
        h = eng.history[1]
        assert eng.novelty_ring is None
        assert h["novelty"] is h["shaped_fitness"] is h["novelty_archive_ids"] is h["novelty_filled"] is None
        logs.append(log.calls)
        states.append((eng.gstate.clone(), {r: eng.pop[r].clone() for r in ROLES},
                       {r: eng.hof[r].clone() for r in ROLES}))
    assert logs[0] == logs[1] and "ga_repopulate" in logs[0]
    assert not any("novelty" in c or "centered_ranks" in c for c in logs[0])
    assert torch.equal(states[0][0], states[1][0])
    for r in ROLES:
        assert torch.equal(states[0][1][r], states[1][1][r]) and torch.equal(states[0][2][r], states[1][2][r])
    sd = eng.state_dict()
    assert sd["ga_novelty"] == {"ga_novelty_weight": 0.0, "ga_novelty_k": None, "ga_novelty_archive": None,
                                "ga_novelty_archive_add": None}
    assert "novelty_ring" not in sd


def test_oracle_ring_bookkeeping_with_several_additions():
    ring = en.Ring(4, np.full(160, -1.0, np.float32))
    assert (ring.head, ring.filled) == (1, 1)
    gn.append(ring, np.arange(3, dtype=np.float32)[:, None] * np.ones(160, np.float32))    # slots 1, 2, 3
    assert (ring.head, ring.filled) == (0, 4)
    gn.append(ring, np.array([7.0, 8.0], np.float32)[:, None] * np.ones(160, np.float32))  # slots 0, 1
    assert (ring.head, ring.filled) == (2, 4)
    assert ring.rows[:, 0].tolist() == [7.0, 8.0, 1.0, 2.0]


@pytest.mark.parametrize("w", [1.0, 0.5], ids=["novelty", "equal"])
def test_engine_follows_the_oracle(w):
    """A = 4, m = 3 over 4 generations (the ring wraps): every generation's novelty (members against the rest of
    the population and the ring as it stood), the selection fitness F, the elites, the fitness-best Hall-of-Fame
    and evaluation row, the drawn archive ids, the rings, head and filled, against the oracle."""
    from coevonet_b200 import layout
    P, A, k, m, E = 6, 4, 3, 3, 2
    eng = _engine(P, ga_novelty_weight=w, ga_novelty_k=k, ga_novelty_archive=A, ga_novelty_archive_add=m)
    _, _, founder = _rows(P)
    obs = {r: en.probe_obs(en.probe_states(99), r) for r in ROLES}
    for r in ROLES:
        assert np.array_equal(eng.novelty_probe_obs[r].numpy(), obs[r])
    rings = {r: en.Ring(A, en.bc(founder[r].numpy()[None, :layout.fc_dim(layout.OBS_DIM[r])], layout.OBS_DIM[r],
                                 obs[r])[0]) for r in ROLES}
    for i, r in enumerate(ROLES):
        assert np.array_equal(eng.novelty_ring[i].numpy(), rings[r].rows)
    for g in range(4):
        before = {r: eng.pop[r].numpy().copy() for r in ROLES}
        filled = rings[ROLES[0]].filled
        eng.step()
        h = eng.history[g]
        assert h["novelty_filled"] == filled
        for i, r in enumerate(ROLES):
            in_dim = layout.OBS_DIM[r]
            dim = layout.fc_dim(in_dim)
            bcs = en.bc(before[r][:, :dim], in_dim, obs[r])
            N = gn.novelty(bcs, 0, bcs, rings[r].rows[:filled], k)
            assert np.array_equal(h["novelty"][r], N), (g, r)
            R = h["fitness"][r]
            F = en.combine(oes.centered_ranks(R), oes.centered_ranks(N), w)
            assert np.array_equal(h["shaped_fitness"][r], F), (g, r)
            ids = ga_es.select_topk(F, E, 1)                 # reference_compat: the reference's tie order
            assert np.array_equal(h["elite_ids"][r], ids), (g, r)
            best = ga_es.select_topk(R, 1, 1)[0]
            assert np.array_equal(eng.hof[r][-1].numpy(), before[r][best]), (g, r)
            assert np.array_equal(eng.best_rows[r].numpy(), before[r][best])
            assert np.array_equal(eng.pop[r][0].numpy(), before[r][ids[0]])      # row 0: the F-best, unmutated
            drawn = gn.draw_ids(99, g, r, m, P)
            assert np.array_equal(h["novelty_archive_ids"][r], drawn), (g, r)
            gn.append(rings[r], bcs[drawn])
            assert np.array_equal(eng.novelty_ring[i].numpy(), rings[r].rows), (g, r)
        assert (eng.novelty_head, eng.novelty_filled) == (rings[ROLES[0]].head, rings[ROLES[0]].filled)
    assert eng.novelty_filled == A


def test_novelty_changes_the_selection():
    """w = 1 selects on the novelty ranks alone: on these rows other elites than the fitness's."""
    a = _engine(6)
    b = _engine(6, ga_novelty_weight=1.0)
    a.step()
    b.step()
    for r in ROLES:
        assert np.array_equal(a.history[0]["fitness"][r], b.history[0]["fitness"][r])
        assert np.array_equal(b.history[0]["shaped_fitness"][r], oes.centered_ranks(b.history[0]["novelty"][r]))
        assert torch.equal(a.hof[r], b.hof[r])                 # the Hall of Fame still takes the fitness-best
    assert any(not np.array_equal(a.history[0]["elite_ids"][r], b.history[0]["elite_ids"][r]) for r in ROLES)


def test_resume_equals_uninterrupted_run(tmp_path):
    kw = dict(NOV, record_history=False)
    full = _engine(5, **kw)
    for _ in range(4):
        full.step(sync=False)
    first = _engine(5, **kw)
    for _ in range(2):
        first.step(sync=False)
    torch.save(first.state_dict(), tmp_path / "nov.pt")
    second = _engine(5, **kw)
    second.load_state_dict(torch.load(tmp_path / "nov.pt", weights_only=False))
    for _ in range(2):
        second.step(sync=False)
    assert torch.equal(second.gstate, full.gstate)
    assert torch.equal(second.novelty_ring, full.novelty_ring)
    assert (second.novelty_head, second.novelty_filled) == (full.novelty_head, full.novelty_filled)
    for r in ROLES:
        assert torch.equal(second.pop[r], full.pop[r]) and torch.equal(second.hof[r], full.hof[r])
        assert torch.equal(second.novelty[r], full.novelty[r])
        assert torch.equal(second.shaped_fitness[r], full.shaped_fitness[r])


def test_resume_refuses_other_novelty_settings():
    nov = _engine(4, record_history=False, **NOV)
    nov.step(sync=False)
    sd = nov.state_dict()
    assert sd["ga_novelty"] == {"ga_novelty_weight": 0.5, "ga_novelty_k": 3, "ga_novelty_archive": 4,
                                "ga_novelty_archive_add": 2}
    assert (sd["novelty_head"], sd["novelty_filled"]) == (3, 3) and tuple(sd["novelty_ring"].shape) == (3, 4, 160)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False).load_state_dict(sd)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **dict(NOV, ga_novelty_archive_add=1)).load_state_dict(sd)
    plain = _engine(4, record_history=False)
    plain.step(sync=False)
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **NOV).load_state_dict(plain.state_dict())
    # a checkpoint without the settings (written before they existed) loads as off
    old = plain.state_dict()
    del old["ga_novelty"]
    fresh = _engine(4, record_history=False)
    fresh.load_state_dict(old)
    for r in ROLES:
        assert torch.equal(fresh.pop[r], plain.pop[r])
    with pytest.raises(ValueError, match="novelty"):
        _engine(4, record_history=False, **NOV).load_state_dict(old)


def _run(rank, world, P, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    torch.set_num_threads(1)
    if world > 1:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from coevonet_b200 import engine
    comm = engine.Comm()
    eng = _engine(P, comm=comm, **NOV)
    evs = [eng.step() for _ in range(3)]
    rec = {key: np.stack([eng.history[g][key][r] for g in range(3) for r in ROLES])
           for key in ("fitness", "novelty", "shaped_fitness", "elite_ids", "novelty_archive_ids")}
    q.put(dict(rank=rank, evs=np.asarray(evs), row0=eng.shard.row0, n_local=eng.shard.n_local,
               ring=eng.novelty_ring.numpy().copy(), hof=np.concatenate([eng.hof[r].numpy() for r in ROLES], axis=1),
               pop=np.concatenate([eng.pop[r].numpy()[:, :1000] for r in ROLES], axis=1), **rec))
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
def test_novelty_two_ranks_match_one_rank():
    """P = 5 over two ranks is 3 + 2 rows: the characterisation all-gather, the per-rank ranks, the F all-gather and
    the extra elite row give the single-rank values; the rings are replicated without a collective."""
    P = 5
    single = _launch(1, P, 29681)[0]
    two = _launch(2, P, 29682)
    for o in two:
        for key in ("novelty", "shaped_fitness", "elite_ids", "novelty_archive_ids", "ring", "hof"):
            assert np.array_equal(o[key], single[key]), key
        np.testing.assert_allclose(o["fitness"], single["fitness"], rtol=1e-12, atol=0)
        np.testing.assert_allclose(o["evs"], single["evs"], rtol=1e-12)
        sl = slice(o["row0"], o["row0"] + o["n_local"])
        assert np.array_equal(o["pop"], single["pop"][sl])
