"""Device-resident Co-GA / Co-ES engines behind the reference's train loops.

One process per GPU.  The population of each role is a ``float32[n_local,
pitch]`` tensor holding the contiguous row block ``[row0, row0 + n_local)`` of
this rank (SURVEY.md section 8e); Hall-of-Fame rows, ES base vectors and the
generation state are replicated.  Collectives (NCCL on GPUs, gloo in the CPU
tests) appear only where the path has an exchange step:

* one all-gather per generation of the per-member fitness (and fitness-sharing
  distances) of the three roles,
* an all-reduce that assembles the elite rows on every rank (each elite row is
  contributed by its owner, zeros elsewhere) -- this is the HoF broadcast,
* one all-reduce of the three roles' ES update ``delta``.

A generation is issued without a host round trip (SURVEY.md 8f N1): the mutation
powers, the evaluation-reward history, the early-stopping counters and the
generation counter live in a device array (``cev_generation_end_f64``), kernels
read sigma from it, elite indices stay on the device, and the non-finite status
word is copied back asynchronously and examined two generations later (so the host
runs one generation ahead of the device).
``step()`` reads the evaluation triple back (one sync) only when asked to.

Everything numeric goes through ``self.k`` -- by default ``coevonet_b200.ops``
(the CUDA kernels).  Tests may inject a checker backend with the same call
signatures to exercise the sharding logic without a GPU; the product never does.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, layout
from .utils import mpe_spec

ROLES = layout.ROLES                    # ("agent_0", "agent_1", "adversary_0")
N_EVAL_GAMES = 10                       # genetic_algorithm.py:18, evolutionary_strategy.py:28
HIST_MIN_CAPACITY = 1024


# ---------------------------------------------------------------------------
# sharding + collectives
# ---------------------------------------------------------------------------
class Shard:
    """Contiguous block partition of P rows over `world` ranks."""

    def __init__(self, P, rank=0, world=1):
        self.P, self.rank, self.world = int(P), int(rank), int(world)
        base, rem = divmod(self.P, self.world)
        self.counts = [base + (1 if r < rem else 0) for r in range(self.world)]
        self.offsets = [sum(self.counts[:r]) for r in range(self.world)]
        self.row0 = self.offsets[self.rank]
        self.n_local = self.counts[self.rank]

    def owner(self, row):
        for r in range(self.world):
            if row < self.offsets[r] + self.counts[r]:
                return r
        raise IndexError(row)


class Comm:
    """torch.distributed when initialised with world_size > 1, otherwise a no-op."""

    def __init__(self, group=None):
        self.enabled = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.group = group
        self.rank = dist.get_rank(group) if self.enabled else 0
        self.world = dist.get_world_size(group) if self.enabled else 1

    def all_gather_rows(self, local, shard):
        """local [n_local, ...] -> [P, ...] in global row order: ONE collective into one tensor
        (uneven shards are padded to the largest block)."""
        return self.all_gather_rows_start(local, shard)()

    def all_gather_rows_start(self, local, shard):
        """Start that collective and return ``finish() -> gathered tensor``: work issued between the two calls
        (on the current stream) overlaps the collective and, more to the point, the wait for the slowest rank."""
        if not self.enabled:
            return lambda: local
        nmax = max(shard.counts)
        tail = tuple(local.shape[1:])
        if local.shape[0] == nmax:
            pad = local.contiguous()
        else:
            pad = torch.zeros((nmax,) + tail, dtype=local.dtype, device=local.device)
            pad[:local.shape[0]] = local
        out = torch.empty((self.world * nmax,) + tail, dtype=local.dtype, device=local.device)
        work = dist.all_gather_into_tensor(out, pad, group=self.group, async_op=True)

        def finish(out=out, pad=pad):
            work.wait()               # NCCL: the current stream waits, the host does not
            if shard.P == self.world * nmax:
                return out
            o = out.view((self.world, nmax) + tail)
            return torch.cat([o[r, :shard.counts[r]] for r in range(self.world)], dim=0)

        return finish

    def all_reduce_sum(self, t):
        if self.enabled:
            dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def all_reduce_max(self, t):
        if self.enabled:
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
        return t

    def broadcast0(self, t):
        """Rank 0's copy of a replicated tensor, on every rank (in place)."""
        if self.enabled:
            dist.broadcast(t, src=dist.get_global_rank(self.group, 0) if self.group is not None else 0,
                           group=self.group)
        return t


def sync_torch_rng(comm, device="cpu"):
    """Give every rank rank 0's torch CPU generator state, so that founders built from the global
    generator (``create_agent`` -> ``nn.Linear`` default init) are identical on all ranks without
    changing what rank 0 -- or a single-process run -- draws."""
    if not comm.enabled:
        return
    state = torch.get_rng_state()
    dev = torch.device(device)
    buf = state.to(dev) if dev.type == "cuda" else state.clone()
    comm.broadcast0(buf)
    torch.set_rng_state(buf.cpu())


#: the opt-in Co-ES update options (Salimans et al. 2017) and their defaults, which run the reference's update
ES_OPTION_DEFAULTS = {"mirrored_sampling": False, "fitness_shaping": "none", "es_optimizer": "sgd", "l2_coeff": 0.0}


def es_options(args, algorithm=None):
    """The Co-ES update options of ``args`` (an absent attribute is its default), validated: ``ValueError`` for an
    unknown value, for mirrored sampling with an odd population and for any non-default option with the GA
    (``algorithm``, or ``args.algorithm`` when not given)."""
    opts = {k: getattr(args, k, d) for k, d in ES_OPTION_DEFAULTS.items()}
    opts["mirrored_sampling"] = bool(opts["mirrored_sampling"])
    opts["l2_coeff"] = float(opts["l2_coeff"])
    if opts["fitness_shaping"] not in ("none", "centered_rank"):
        raise ValueError(f"fitness_shaping must be 'none' or 'centered_rank', not {opts['fitness_shaping']!r}")
    if opts["es_optimizer"] not in ("sgd", "adam"):
        raise ValueError(f"es_optimizer must be 'sgd' or 'adam', not {opts['es_optimizer']!r}")
    if not np.isfinite(opts["l2_coeff"]) or opts["l2_coeff"] < 0:
        raise ValueError(f"l2_coeff must be a finite number >= 0, not {opts['l2_coeff']}")
    if opts != ES_OPTION_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) == "GA":
        changed = sorted(k for k in opts if opts[k] != ES_OPTION_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-ES options, not available with --algorithm GA")
    if opts["mirrored_sampling"] and int(args.population) % 2:
        raise ValueError(f"mirrored sampling needs an even population, not {args.population}")
    return opts


#: the Co-ES search distribution and its default: one isotropic Gaussian per role (the reference), separable NES
#: (a per-parameter mutation strength, Schaul et al. 2011) or LM-MA-ES (limited-memory matrix adaptation, Loshchilov
#: et al. 2019); sigma_learning_rate None = default_sigma_learning_rate; es_lmma_memory None = LMMA_DEFAULT_MEMORY
#: with lmma, and only then part of the settings (so the settings of the other distributions keep their two keys)
ES_DISTRIBUTION_DEFAULTS = {"es_distribution": "isotropic", "sigma_learning_rate": None}
#: LM-MA-ES direction vectors per role.  Not the paper's 4 + floor(3 ln n) = 39: vector j moves at c_c,j = lam / (4^j n),
#: so at lam = 1024 and n ~ 138 k vector 5 reaches ~14 % of its stationary norm in 1e4 generations and vector 7 < 1 %;
#: vectors past ~8 cost a K5 term each and contribute nothing in runs of this size
LMMA_DEFAULT_MEMORY = 8
#: the fewest Linear entries of a role's row (the adversary's): LM-MA-ES needs c_sigma = 2 lam / n < 1 for every role
LMMA_MIN_DIM = min(len(layout.fc_perturbable_index(d)) for d in set(layout.OBS_DIM.values()))


def es_distribution(args, algorithm=None):
    """The Co-ES search distribution settings of ``args`` (an absent attribute is its default), validated:
    ``ValueError`` for an unknown distribution, for any non-default setting with the GA, for ``separable`` with
    Adam, L2 weight decay or ``--adaptive`` (they would fight the per-parameter step) and for a
    ``sigma_learning_rate`` that is not a finite number > 0 or is given without ``separable``."""
    opts = {k: getattr(args, k, d) for k, d in ES_DISTRIBUTION_DEFAULTS.items()}
    memory = getattr(args, "es_lmma_memory", None)
    if opts["es_distribution"] not in ("isotropic", "separable", "lmma"):
        raise ValueError(f"es_distribution must be 'isotropic', 'separable' or 'lmma', not {opts['es_distribution']!r}")
    if opts != ES_DISTRIBUTION_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) == "GA":
        changed = sorted(k for k in opts if opts[k] != ES_DISTRIBUTION_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-ES options, not available with --algorithm GA")
    separable = opts["es_distribution"] == "separable"
    if opts["sigma_learning_rate"] is not None:
        opts["sigma_learning_rate"] = float(opts["sigma_learning_rate"])
        if not separable:
            raise ValueError("sigma_learning_rate needs es_distribution 'separable'")
        if not np.isfinite(opts["sigma_learning_rate"]) or opts["sigma_learning_rate"] <= 0:
            raise ValueError(f"sigma_learning_rate must be a finite number > 0, not {opts['sigma_learning_rate']}")
    if separable:
        if getattr(args, "es_optimizer", "sgd") != "sgd" or float(getattr(args, "l2_coeff", 0.0)) != 0.0:
            raise ValueError("es_distribution 'separable' takes its own step: not available with es_optimizer "
                             "'adam' or a nonzero l2_coeff")
        if getattr(args, "adaptive", False):
            raise ValueError("es_distribution 'separable' adapts every sigma itself: not available with --adaptive")
    if memory is not None and opts["es_distribution"] != "lmma":
        raise ValueError("es_lmma_memory needs es_distribution 'lmma'")
    if opts["es_distribution"] == "lmma":
        opts["es_lmma_memory"] = memory
        _lmma_refusals(args, opts)
    return opts


def _lmma_refusals(args, opts):
    """The settings LM-MA-ES refuses (``ValueError``), and its memory m resolved into ``opts``."""
    m = LMMA_DEFAULT_MEMORY if opts["es_lmma_memory"] is None else int(opts["es_lmma_memory"])
    if not 1 <= m <= _lib.SUBSPACE_MAX_DIM:
        raise ValueError(f"es_lmma_memory must be in [1, {_lib.SUBSPACE_MAX_DIM}], not {m}")
    opts["es_lmma_memory"] = m
    if getattr(args, "es_optimizer", "sgd") != "sgd" or float(getattr(args, "l2_coeff", 0.0)) != 0.0:
        raise ValueError("es_distribution 'lmma' takes its own step: not available with es_optimizer 'adam' or a "
                         "nonzero l2_coeff")
    if getattr(args, "adaptive", False):
        raise ValueError("es_distribution 'lmma' adapts sigma by cumulative step-size adaptation: not available with "
                         "--adaptive")
    if getattr(args, "fitness_shaping", "none") != "none":
        raise ValueError("es_distribution 'lmma' weights the ranked members with its own log weights: not available "
                         "with fitness_shaping 'centered_rank'")
    if getattr(args, "mirrored_sampling", False):
        raise ValueError("es_distribution 'lmma': mirrored pairs under truncation selection bias the step-size "
                         "adaptation; not available with mirrored sampling")
    if int(getattr(args, "es_subspace_dim", 0) or 0):
        raise ValueError("es_distribution 'lmma' has its own search shape: not available with es_subspace_dim")
    if float(getattr(args, "es_novelty_weight", 0.0) or 0.0):
        raise ValueError("es_distribution 'lmma' recombines on the fitness: not available with es_novelty_weight")
    P = int(getattr(args, "population", 2))
    if P < 2:
        raise ValueError(f"es_distribution 'lmma' selects the best half: needs a population >= 2, not {P}")
    if 2 * P >= LMMA_MIN_DIM:
        raise ValueError(f"es_distribution 'lmma' needs c_sigma = 2 population / n < 1: population {P} is too large "
                         f"for n = {LMMA_MIN_DIM}")


def lmma_constants(lam, n, m):
    """LM-MA-ES's constants (Loshchilov, Glasmachers & Beyer 2019, Algorithm 1) for population lam, dimension n and m
    vectors, fp64: mu = lam // 2, the log weights w_i = (ln(mu + 1/2) - ln(i + 1)) / sum_j (...) for i < mu,
    mu_w = 1 / sum w_i^2, c_sigma = 2 lam / n, c_d,j = 1 / (1.5^j n), c_c,j = lam / (4^j n) for j < m, and alpha_k =
    prod_{j < k} (1 - c_d,j) for k <= m (the coefficient of z after k transform steps)."""
    mu = int(lam) // 2
    raw = np.array([np.log(mu + 0.5) - np.log(i + 1) for i in range(mu)], dtype=np.float64)
    w = raw / raw.sum()
    c_d = [1.0 / (1.5 ** j * n) for j in range(m)]
    alpha = [1.0]
    for j in range(m):
        alpha.append(alpha[-1] * (1.0 - c_d[j]))
    return {"mu": mu, "w": w, "mu_w": float(1.0 / np.sum(w * w)), "c_sigma": 2.0 * lam / n, "c_d": c_d,
            "c_c": [lam / (4.0 ** j * n) for j in range(m)], "alpha": alpha}


#: the Co-ES Hall of Fame and its defaults: 0 = off (every member plays the other roles' current base agents only)
ES_HOF_DEFAULTS = {"es_hof_size": 0, "es_hof_opponents": 1}


def es_hof(args, algorithm=None):
    """The Co-ES Hall-of-Fame settings of ``args`` (an absent attribute is its default), validated: ``ValueError``
    for a negative archive size H, for K opponent sets outside [1, H] when H > 0, for K other than 1 when H = 0 and
    for any non-default setting with the GA (which keeps its own Hall of Fame, ``--hof_size``)."""
    opts = {k: int(getattr(args, k, d)) for k, d in ES_HOF_DEFAULTS.items()}
    H, K = opts["es_hof_size"], opts["es_hof_opponents"]
    if opts != ES_HOF_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) == "GA":
        raise ValueError("es_hof_size, es_hof_opponents: Co-ES options, not available with --algorithm GA "
                         "(the GA keeps its own Hall of Fame, --hof_size)")
    if H < 0:
        raise ValueError(f"es_hof_size must be >= 0, not {H}")
    if H == 0 and K != 1:
        raise ValueError(f"es_hof_opponents {K} needs an archive: es_hof_size must be >= {max(K, 1)}")
    if H > 0 and not 1 <= K <= H:
        raise ValueError(f"es_hof_opponents must be in [1, es_hof_size = {H}], not {K}")
    return opts


#: Co-ES guided search in the subspace of the last k update estimates and its defaults: 0 = off (the isotropic
#: search); es_subspace_alpha None = the default share 0.5 of the variance outside the subspace when k > 0
ES_SUBSPACE_DEFAULTS = {"es_subspace_dim": 0, "es_subspace_alpha": None}
SUBSPACE_DEFAULT_ALPHA = 0.5


def es_subspace(args, algorithm=None):
    """The Co-ES guided-search settings of ``args`` (an absent attribute is its default), validated: ``ValueError``
    for any non-default setting with the GA, for a subspace dimension k outside [0, 32], for an alpha outside (0, 1]
    or given while k = 0, and for k > 0 together with ``separable`` search or ``--regenerate_noise`` (the regenerated
    update would need the subspace term too).  With k > 0 an alpha left unset becomes 0.5."""
    opts = {k: getattr(args, k, d) for k, d in ES_SUBSPACE_DEFAULTS.items()}
    if opts != ES_SUBSPACE_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) == "GA":
        changed = sorted(k for k in opts if opts[k] != ES_SUBSPACE_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-ES options, not available with --algorithm GA")
    k = int(opts["es_subspace_dim"])
    if not 0 <= k <= _lib.SUBSPACE_MAX_DIM:
        raise ValueError(f"es_subspace_dim must be in [0, {_lib.SUBSPACE_MAX_DIM}], not {k}")
    alpha = opts["es_subspace_alpha"]
    if alpha is not None:
        alpha = float(alpha)
        if k == 0:
            raise ValueError("es_subspace_alpha needs es_subspace_dim > 0")
        if not 0.0 < alpha <= 1.0:
            raise ValueError(f"es_subspace_alpha must be in (0, 1], not {alpha}")
    if k:
        if getattr(args, "es_distribution", "isotropic") != "isotropic":
            raise ValueError("es_subspace_dim: guided search is not available with es_distribution "
                             f"{getattr(args, 'es_distribution', 'isotropic')!r}")
        if not getattr(args, "update_from_members", True):
            raise ValueError("es_subspace_dim: guided search needs the update from the members, not available with "
                             "--regenerate_noise")
        alpha = SUBSPACE_DEFAULT_ALPHA if alpha is None else alpha
    return {"es_subspace_dim": k, "es_subspace_alpha": alpha}


#: Co-ES novelty search (NS-ES / NSR-ES, Conti et al. 2018) and its defaults: weight 0 = off (the fitness is the
#: reward); es_novelty_k / es_novelty_archive None = NOVELTY_DEFAULT_K / NOVELTY_DEFAULT_ARCHIVE when the weight is > 0
ES_NOVELTY_DEFAULTS = {"es_novelty_weight": 0.0, "es_novelty_k": None, "es_novelty_archive": None}
NOVELTY_DEFAULT_K, NOVELTY_DEFAULT_ARCHIVE = 10, 1024
#: Philox stream of the novelty search's probe world states (cev_init_states_f64): apart from the training states
#: (role + 4 * gen), the evaluation games (0x40000000 + gen) and the Hall-of-Fame matrix (0x50000000)
NOVELTY_PROBE_TAG = 0x60000000


def es_novelty(args, algorithm=None):
    """The Co-ES novelty-search settings of ``args`` (an absent attribute is its default), validated: ``ValueError``
    for any non-default setting with the GA, for a weight w outside [0, 1], for k or the archive size given while
    w = 0, for k outside [1, 32], for an archive size outside [1, 32768] and for w > 0 without centered-rank fitness
    shaping (the reward and the novelty are combined as ranks).  With w > 0 an unset k becomes 10 and an unset
    archive size 1024."""
    opts = {k: getattr(args, k, d) for k, d in ES_NOVELTY_DEFAULTS.items()}
    if opts != ES_NOVELTY_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) == "GA":
        changed = sorted(k for k in opts if opts[k] != ES_NOVELTY_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-ES options, not available with --algorithm GA")
    w = float(opts["es_novelty_weight"])
    if not 0.0 <= w <= 1.0:
        raise ValueError(f"es_novelty_weight must be in [0, 1], not {w}")
    if w == 0.0:
        given = [k for k in ("es_novelty_k", "es_novelty_archive") if opts[k] is not None]
        if given:
            raise ValueError(f"{', '.join(given)} needs es_novelty_weight > 0")
        return dict(ES_NOVELTY_DEFAULTS)
    k = NOVELTY_DEFAULT_K if opts["es_novelty_k"] is None else int(opts["es_novelty_k"])
    if not 1 <= k <= _lib.NOVELTY_MAX_K:
        raise ValueError(f"es_novelty_k must be in [1, {_lib.NOVELTY_MAX_K}], not {k}")
    A = NOVELTY_DEFAULT_ARCHIVE if opts["es_novelty_archive"] is None else int(opts["es_novelty_archive"])
    if not 1 <= A <= _lib.NOVELTY_MAX_ARCHIVE:
        raise ValueError(f"es_novelty_archive must be in [1, {_lib.NOVELTY_MAX_ARCHIVE}], not {A}")
    if getattr(args, "fitness_shaping", "none") != "centered_rank":
        raise ValueError("es_novelty_weight combines the ranks of the reward and of the novelty: it needs "
                         "fitness_shaping 'centered_rank'")
    return {"es_novelty_weight": w, "es_novelty_k": k, "es_novelty_archive": A}


#: Co-GA novelty search (Lehman & Stanley 2011) and its defaults: weight 0 = off (selection on the fitness); the
#: others None = GA_NOVELTY_DEFAULT_K / _ARCHIVE / _ADD when the weight is > 0
GA_NOVELTY_DEFAULTS = {"ga_novelty_weight": 0.0, "ga_novelty_k": None, "ga_novelty_archive": None,
                       "ga_novelty_archive_add": None}
GA_NOVELTY_DEFAULT_K, GA_NOVELTY_DEFAULT_ARCHIVE, GA_NOVELTY_DEFAULT_ADD = 10, 1024, 1


def ga_novelty(args, algorithm=None):
    """The Co-GA novelty-search settings of ``args`` (an absent attribute is its default), validated: ``ValueError``
    for any non-default setting with the ES, for a weight w outside [0, 1] (NaN included), for k, the archive size A
    or the archive additions m given while w = 0, for k outside [1, 32], for A outside [1, 32768] and for m outside
    [1, A].  With w > 0 an unset k becomes 10, A 1024 and m 1."""
    opts = {k: getattr(args, k, d) for k, d in GA_NOVELTY_DEFAULTS.items()}
    if opts != GA_NOVELTY_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) != "GA":
        changed = sorted(k for k in opts if opts[k] != GA_NOVELTY_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-GA options, not available with --algorithm ES")
    w = float(opts["ga_novelty_weight"])
    if not 0.0 <= w <= 1.0:
        raise ValueError(f"ga_novelty_weight must be in [0, 1], not {w}")
    if w == 0.0:
        given = [k for k in ("ga_novelty_k", "ga_novelty_archive", "ga_novelty_archive_add") if opts[k] is not None]
        if given:
            raise ValueError(f"{', '.join(given)} needs ga_novelty_weight > 0")
        return dict(GA_NOVELTY_DEFAULTS)
    k = GA_NOVELTY_DEFAULT_K if opts["ga_novelty_k"] is None else int(opts["ga_novelty_k"])
    if not 1 <= k <= _lib.NOVELTY_MAX_K:
        raise ValueError(f"ga_novelty_k must be in [1, {_lib.NOVELTY_MAX_K}], not {k}")
    A = GA_NOVELTY_DEFAULT_ARCHIVE if opts["ga_novelty_archive"] is None else int(opts["ga_novelty_archive"])
    if not 1 <= A <= _lib.NOVELTY_MAX_ARCHIVE:
        raise ValueError(f"ga_novelty_archive must be in [1, {_lib.NOVELTY_MAX_ARCHIVE}], not {A}")
    m = GA_NOVELTY_DEFAULT_ADD if opts["ga_novelty_archive_add"] is None else int(opts["ga_novelty_archive_add"])
    if not 1 <= m <= A:
        raise ValueError(f"ga_novelty_archive_add must be in [1, ga_novelty_archive = {A}], not {m}")
    return {"ga_novelty_weight": w, "ga_novelty_k": k, "ga_novelty_archive": A, "ga_novelty_archive_add": m}


#: Co-GA safe mutations through output gradients (SM-G-SUM, Lehman et al. 2018) and their defaults: off; with the
#: option on, an unset floor becomes GA_SAFE_MUTATION_DEFAULT_FLOOR (no mutation is amplified more than 100x)
GA_SAFE_MUTATION_DEFAULTS = {"ga_safe_mutation": False, "ga_safe_mutation_floor": None}
GA_SAFE_MUTATION_DEFAULT_FLOOR = 0.01


def ga_safe_mutation(args, algorithm=None):
    """The Co-GA safe-mutation settings of ``args`` (an absent attribute is its default), validated: ``ValueError``
    for either setting with the ES, for a floor given without ``ga_safe_mutation`` and for a floor that is not finite
    and > 0 (as a float32, the kernel's type).  With the option on an unset floor becomes 0.01."""
    opts = {k: getattr(args, k, d) for k, d in GA_SAFE_MUTATION_DEFAULTS.items()}
    opts["ga_safe_mutation"] = bool(opts["ga_safe_mutation"])
    if opts != GA_SAFE_MUTATION_DEFAULTS and (algorithm or getattr(args, "algorithm", "ES")) != "GA":
        changed = sorted(k for k in opts if opts[k] != GA_SAFE_MUTATION_DEFAULTS[k])
        raise ValueError(f"{', '.join(changed)}: Co-GA options, not available with --algorithm ES")
    if not opts["ga_safe_mutation"]:
        if opts["ga_safe_mutation_floor"] is not None:
            raise ValueError("ga_safe_mutation_floor needs ga_safe_mutation")
        return dict(GA_SAFE_MUTATION_DEFAULTS)
    floor = GA_SAFE_MUTATION_DEFAULT_FLOOR if opts["ga_safe_mutation_floor"] is None \
        else float(opts["ga_safe_mutation_floor"])
    with np.errstate(over="ignore"):
        f32 = np.float32(floor)
    if not (np.isfinite(f32) and f32 > 0):
        raise ValueError(f"ga_safe_mutation_floor must be finite and > 0, not {floor}")
    return {"ga_safe_mutation": True, "ga_safe_mutation_floor": floor}


def default_sigma_learning_rate(d):
    """SNES's sigma learning rate for d parameters, (3 + ln d) / (5 sqrt d) (Schaul et al. 2011), in fp64."""
    return (3.0 + np.log(float(d))) / (5.0 * np.sqrt(float(d)))


def default_kernels():
    from . import ops
    return ops


def _limit_cycles(k, limit):
    return k.cycles_for_limit(limit)


# ---------------------------------------------------------------------------
# shared evaluation plumbing
# ---------------------------------------------------------------------------
class _EngineBase:
    kind = "base"

    def __init__(self, args, device, env=None, kernels=None, comm=None):
        self.args = args
        self.device = torch.device(device)
        self.k = kernels if kernels is not None else default_kernels()
        self.comm = comm if comm is not None else Comm()
        self.env = env if env is not None else mpe_spec.DeviceMPEEnv()
        self.seed = int(getattr(args, "seed", mpe_spec.ENV_SEED))
        self.compat = bool(getattr(args, "reference_compat", True))
        self.E = int(getattr(args, "envs_per_member", 1))
        self.pos_first = bool(getattr(args, "integrate_pos_first", True))
        # "reference": the host PCG64 stream env.reset() consumes upstream (exact episode-for-
        # episode initial states of a reference run); "device": Philox records generated on
        # the GPU (no host RNG work or upload; needed at large P)
        self.init_mode = getattr(args, "init_states", "reference")
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.gen = 0
        #: per-generation records (small runs / tests): filled when args.record_history is set
        self.history = [] if getattr(args, "record_history", False) else None
        #: bench hook: when a list, (start, stop) CUDA events are recorded around every
        #: population K1 launch on the launching stream
        self.k1_events = None
        #: evaluate the three roles of a generation on three CUDA streams (they are independent: every
        #: member plays the OTHER roles' base policies of the previous generation), so one role's kernels
        #: fill the partial waves and launch gaps of another's
        self.overlap_roles = bool(getattr(args, "overlap_roles", True)) and self.device.type == "cuda"
        self._role_streams = None
        self._eval_stream = None
        #: the roles' rollouts of a generation as ONE lockstep pass (cev_mpe_rollout_roles_f32) instead of one pass
        #: per role on three streams: one member kernel and one opponent kernel share the SMs at any time
        self.fused_roles = bool(getattr(args, "fused_roles", True)) and self.device.type == "cuda"
        #: ES update from the materialised members (K6 as an HBM-bound read) instead of regenerating the
        #: noise from the Philox key (K6 as ALU work); both are within fp32 rounding of each other
        self.update_from_members = bool(getattr(args, "update_from_members", True))
        #: selection order (K4): the reference's expression under reference_compat
        self.order = _lib.ORDER_REFERENCE if self.compat else _lib.ORDER_STABLE_DESC
        self.adaptive = bool(getattr(args, "adaptive", False))
        self.early_stopping = bool(getattr(args, "early_stopping", False))
        # ---- generation state on the device (N1) ------------------------------------------------
        self.hist_cap = max(int(getattr(args, "generations", 1)) + 1, HIST_MIN_CAPACITY)
        self.gstate = self.k.generation_state(
            [args.mutation_power_agent_0, args.mutation_power_agent_1, args.mutation_power_adversary],
            self.hist_cap, self.device)
        self._eval_init_tag = 0x40000000
        #: (pinned host copy, event) of the generations whose status word has not been looked at yet, oldest first
        self._pending_status = []

    # -- replicated / sharded state helpers -----------------------------------------------------
    def sigma_dev(self, role):
        """One-element fp64 device view of the role's mutation power (what K3/K5/K6 read)."""
        i = _lib.GS_SIGMA + ROLES.index(role)
        return self.gstate[i:i + 1]

    def sigma(self, role):
        """Host copy of the role's CURRENT mutation power (synchronises)."""
        return float(self.gstate[_lib.GS_SIGMA + ROLES.index(role)].item())

    def rollout_variant(self, P_global, K):
        """K1 kernel variant chosen from the GLOBAL evaluation shape, so a sharded run executes the
        same arithmetic as a single-GPU run of the same population (ADVICE r1)."""
        plan = getattr(self.k, "rollout_plan", None)
        if plan is None or self.device.type != "cuda":
            return 0
        used, _ = plan(self.device.index, int(P_global), int(K), self.E, 25)
        return used

    # initial states of `n_rows` x K x E episodes for the rows [row0, row0+n_local) of a
    # P-row evaluation; in reference mode every rank draws the whole block to keep the
    # host stream in step, then slices its rows.
    def _initial_states(self, P, K, shard, stream_tag):
        E = self.E
        if self.init_mode == "reference":
            block = self.env.draw_initial_states(P * K * E).reshape(P, K, E, mpe_spec.INIT_STATE_DIM)
            mine = block[shard.row0:shard.row0 + shard.n_local]
            return torch.from_numpy(np.ascontiguousarray(mine)).to(self.device)
        rec0 = shard.row0 * K * E
        out = self.k.init_states(self.seed, stream_tag, shard.n_local * K * E, self.device, rec0=rec0)
        return out.reshape(shard.n_local, K, E, mpe_spec.INIT_STATE_DIM)

    # -- status word: examined two generations late, without a sync --------------------------------
    def _post_status(self):
        if self.device.type != "cuda":
            self._pending_status.append((self.status.clone(), None))
            return
        host = torch.empty(1, dtype=torch.int32).pin_memory()
        host.copy_(self.status, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending_status.append((host, ev))

    def _raise_pending_status(self, keep=1):
        """Look at the status words posted so far, except the newest ``keep``.  A generation starts by checking
        the generation BEFORE the previous one: the previous one's copy was enqueued a moment ago, and waiting
        for it would stop the host from running ahead of the device (0.5 ms of idle device per generation)."""
        if self.device.type != "cuda":
            keep = 0
        while len(self._pending_status) > keep:
            host, ev = self._pending_status.pop(0)
            if ev is not None:
                ev.synchronize()      # recorded at least a whole generation ago: complete in steady state
            self.k.raise_on_status(host)

    def check_status(self):
        """Surface device-detected faults now (synchronises): the reference's ``ValueError``."""
        self._raise_pending_status(keep=0)
        self.k.raise_on_status(self.status)

    def _role_slot(self, out, role, limit):
        s0, s1, sadv = self.k.reward_slots(out, agent_step_limit=limit, reference_compat=self.compat)
        return {"agent_0": s0, "agent_1": s1, "adversary_0": sadv}[role]

    # -- end of generation: evaluation games + device bookkeeping ----------------------------------
    def _finish_generation(self, row_a0, row_a1, row_adv):
        """``evaluate_current_weights`` (genetic_algorithm.py:12-29) on the three given rows +
        reward history, adaptive sigma and early-stopping counters, all on the device
        (``cev_generation_end_f64``).  Replicated on every rank.  On CUDA this runs on a side
        stream: the next generation only waits for it when its sigma depends on it."""
        a = self.args
        limit = a.max_evaluation_steps
        if self.init_mode == "reference":
            init = torch.from_numpy(self.env.draw_initial_states(N_EVAL_GAMES)).to(self.device)
        else:
            init = self.k.init_states(self.seed, self._eval_init_tag + self.gen, N_EVAL_GAMES, self.device)
        init = init.reshape(1, 1, N_EVAL_GAMES, mpe_spec.INIT_STATE_DIM)

        def body():
            out = self.k.mpe_rollout("agent_0", row_a0.reshape(1, -1), row_adv.reshape(1, -1),
                                     row_a1.reshape(1, -1), init, n_cycles=_limit_cycles(self.k, limit),
                                     pos_first=self.pos_first, status=self.status)
            self.k.generation_end(out, self.gstate, self.hist_cap, agent_step_limit=limit,
                                  reference_compat=self.compat, adaptive=self.adaptive,
                                  sigma_max=a.max_mutation_power, sigma_min=a.min_mutation_power,
                                  early_stopping=self.early_stopping, min_delta=a.min_delta, patience=a.patience)
            self._post_status()

        if self.device.type == "cuda":
            if self._eval_stream is None:
                # high priority: the evaluation games are one small launch (a 4-CTA cluster) that must find four free
                # SMs among the persistent rollout kernels of the next generation instead of waiting for their end
                self._eval_stream = torch.cuda.Stream(device=self.device, priority=-1)
            main = torch.cuda.current_stream(self.device)
            self._eval_stream.wait_stream(main)
            with torch.cuda.stream(self._eval_stream):
                init.record_stream(self._eval_stream)
                body()
        else:
            body()

    def _join_eval(self):
        """Make the current stream wait for the evaluation games / generation state of the previous
        generation (needed before anything that reads sigma when it adapts, and before host reads)."""
        if self._eval_stream is not None:
            torch.cuda.current_stream(self.device).wait_stream(self._eval_stream)

    def last_eval(self):
        """(agent_0, agent_1, adversary_0) evaluation rewards of the generation just finished
        (synchronises)."""
        self._join_eval()
        v = self.gstate[_lib.GS_LAST_EVAL:_lib.GS_LAST_EVAL + 3].cpu().tolist()
        return tuple(float(x) for x in v)

    def host_state(self):
        """Host copy of the generation state (synchronises): generation count, sigmas, reward and
        sigma histories, early-stopping flag -- what the reference keeps in Python lists."""
        self._join_eval()
        gs = self.gstate.cpu().numpy()
        n = int(gs[_lib.GS_GEN])
        h = gs[_lib.GS_HIST:_lib.GS_HIST + 3 * self.hist_cap].reshape(self.hist_cap, 3)
        sh = gs[_lib.GS_HIST + 3 * self.hist_cap:].reshape(self.hist_cap + 1, 3)
        stop = int(gs[_lib.GS_STOP])
        return {"generations": n, "sigma": {r: float(gs[_lib.GS_SIGMA + i]) for i, r in enumerate(ROLES)},
                "rewards": {r: h[:min(n, self.hist_cap), i].copy() for i, r in enumerate(ROLES)},
                "sigma_history": {r: sh[:min(n, self.hist_cap) + 1, i].copy() for i, r in enumerate(ROLES)},
                "best": {r: float(gs[_lib.GS_BEST + i]) for i, r in enumerate(ROLES)},
                "stale": {r: int(gs[_lib.GS_STALE + i]) for i, r in enumerate(ROLES)},
                "stop_role": ROLES[stop - 1] if stop else None, "stop_generation": int(gs[_lib.GS_STOP_GEN])}

    def write_back_args(self):
        """Mirror the device sigmas into ``args.mutation_power_*`` (the reference mutates ``args``)."""
        s = self.host_state()["sigma"]
        self.args.mutation_power_agent_0 = s["agent_0"]
        self.args.mutation_power_agent_1 = s["agent_1"]
        self.args.mutation_power_adversary = s["adversary_0"]

    def should_stop(self):
        """Early-stopping decision of the generation just finished (synchronises; identical on all
        ranks, max-reduced anyway so control flow cannot diverge)."""
        self._join_eval()
        flag = self.gstate[_lib.GS_STOP:_lib.GS_STOP + 1].clone()
        self.comm.all_reduce_max(flag)
        return int(flag.item())

    def _run_roles(self, fn):
        """Run ``fn(role)`` for the three roles, on three CUDA streams when enabled."""
        if self.overlap_roles and self.k1_events is None:
            if self._role_streams is None:
                self._role_streams = [torch.cuda.Stream(device=self.device) for _ in ROLES]
            main = torch.cuda.current_stream(self.device)
            for role, st in zip(ROLES, self._role_streams):
                st.wait_stream(main)
                with torch.cuda.stream(st):
                    fn(role)
            for st in self._role_streams:
                main.wait_stream(st)
        else:
            for role in ROLES:
                fn(role)

    def _rollouts(self, specs, limit):
        """K1 for the given (role, members, opp_a, opp_b, init) specs -> {role: out fp64 [n_local, K, E, 4]}."""
        n_cycles = _limit_cycles(self.k, limit)
        if self.fused_roles and self.k1_events is None and hasattr(self.k, "mpe_rollout_roles") and len(specs) > 1:
            outs = self.k.mpe_rollout_roles(specs, n_cycles=n_cycles, pos_first=self.pos_first, status=self.status,
                                            variant=self.variant)
            return {spec[0]: out for spec, out in zip(specs, outs)}
        res = {}

        def one(role):
            spec = next(sp for sp in specs if sp[0] == role)
            if self.k1_events is not None:
                e0 = torch.cuda.Event(enable_timing=True)
                e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
            res[role] = self.k.mpe_rollout(role, spec[1], spec[2], spec[3], spec[4], n_cycles=n_cycles,
                                           pos_first=self.pos_first, status=self.status, variant=self.variant)
            if self.k1_events is not None:
                e1.record()
                self.k1_events.append((e0, e1))

        self._run_roles(one)
        return res

    # -- checkpoint / resume (N2) ---------------------------------------------------------------
    def _base_state(self):
        self._join_eval()
        return {"kind": self.kind, "gen": self.gen, "seed": self.seed, "P": self.P, "world": self.comm.world,
                "row0": self.shard.row0, "n_local": self.shard.n_local, "hist_cap": self.hist_cap,
                "gstate": self.gstate.cpu(), "env": self.env.state_dict() if hasattr(self.env, "state_dict") else None}

    def _load_base_state(self, sd):
        if sd["kind"] != self.kind:
            raise ValueError(f"checkpoint holds a {sd['kind']} engine, this is {self.kind}")
        if int(sd["P"]) != self.P:
            raise ValueError(f"checkpoint population {sd['P']} != {self.P}")
        if int(sd["seed"]) != self.seed:
            raise ValueError("checkpoint was written with another seed")
        self.gen = int(sd["gen"])
        gs = sd["gstate"].to(torch.float64)
        if int(sd["hist_cap"]) != self.hist_cap:          # re-home the histories in this run's capacity
            old = int(sd["hist_cap"])
            new = self.k.generation_state([0, 0, 0], self.hist_cap, "cpu")
            new[:_lib.GS_HIST] = gs[:_lib.GS_HIST]
            n = min(old, self.hist_cap)
            new[_lib.GS_HIST:_lib.GS_HIST + 3 * n] = gs[_lib.GS_HIST:_lib.GS_HIST + 3 * n]
            so, sn = _lib.GS_HIST + 3 * old, _lib.GS_HIST + 3 * self.hist_cap
            new[sn:sn + 3 * (n + 1)] = gs[so:so + 3 * (n + 1)]
            gs = new
        self.gstate.copy_(gs.to(self.device))
        if sd.get("env") is not None and hasattr(self.env, "load_state_dict"):
            self.env.load_state_dict(sd["env"])
        self._pending_status = []


# ---------------------------------------------------------------------------
# Co-GA  (genetic_algorithm.py:51-374)
# ---------------------------------------------------------------------------
class GAEngine(_EngineBase):
    """State: per role the sharded population, the replicated HoF ring
    (oldest first, like the reference's list) and the frozen founder row the
    reference measures diversity against (Appendix C #3).

    Opt-in novelty search (``ga_novelty``): a member's behaviour characterisation is the ES novelty search's (its
    softmax action distributions on 32 probe observations drawn once from the seed), fp32 [160].  Per role a ring
    ``novelty_ring`` fp32 [A, 160], replicated, starts with the founder's and receives m drawn members'
    characterisations after every selection.  A member's novelty is the mean distance to its k nearest among the
    other members and the archive (``cev_ga_novelty_knn_f64``); parents are selected on F = (1 - w) cr(fitness) +
    w cr(novelty) (cr: centered ranks of the global vectors), while the Hall of Fame and the evaluation games take
    the fitness-best member.

    Opt-in safe mutations (``ga_safe_mutation``, SM-G-SUM): after the elite all-reduce every rank computes the scale
    rows of the E elites on the same probe observations (``cev_ga_safe_scale_f32``; deterministic, so replicated
    without a collective), and K3 multiplies each parameter's fl(sigma z) by the scale of the elite it came from."""

    kind = "GA"

    def __init__(self, args, device, pop_rows, hof_rows, founder_rows, env=None, kernels=None, comm=None):
        super().__init__(args, device, env, kernels, comm)
        self.P = int(args.population)
        es_options(args, "GA")                           # refuses the Co-ES options
        es_distribution(args, "GA")
        es_hof(args, "GA")
        es_subspace(args, "GA")
        es_novelty(args, "GA")
        self.novelty_opts = ga_novelty(args, "GA")
        self.safe_opts = ga_safe_mutation(args, "GA")
        #: safe mutations (SM-G-SUM): on / off, and the floor of the sensitivity
        self.safe = self.safe_opts["ga_safe_mutation"]
        self.safe_floor = self.safe_opts["ga_safe_mutation_floor"]
        #: this generation's scale rows per role, fp32 [E, pitch] (``ga_safe_scale`` of the elites)
        self.safe_scale = {r: None for r in ROLES}
        #: novelty weight w (0: off), nearest neighbours k, archive capacity A and additions per generation m
        self.novelty_w = self.novelty_opts["ga_novelty_weight"]
        self.novelty_k = self.novelty_opts["ga_novelty_k"]
        self.novelty_A = self.novelty_opts["ga_novelty_archive"]
        self.novelty_m = self.novelty_opts["ga_novelty_archive_add"]
        self.shard = Shard(self.P, self.comm.rank, self.comm.world)
        self.pop = {r: pop_rows[r].to(self.device).contiguous() for r in ROLES}       # [n_local, pitch]
        self.hof = {r: hof_rows[r].to(self.device).contiguous() for r in ROLES}       # [hof, pitch]
        self.founder = {r: founder_rows[r].to(self.device).contiguous() for r in ROLES}
        # replicated state is rank 0's, whatever each rank's generator produced (ADVICE r1)
        for r in ROLES:
            self.comm.broadcast0(self.hof[r])
            self.comm.broadcast0(self.founder[r])
        self.elites = {r: None for r in ROLES}
        self.elite_ids = {r: None for r in ROLES}
        #: the row the Hall of Fame and the evaluation games take: elites[0], or with novelty the fitness-best member
        self.best_rows = {r: None for r in ROLES}
        self.fitness = {r: None for r in ROLES}
        self.diversity = {r: None for r in ROLES}       # 0-dim device tensors
        self.novelty_ring = self.novelty_probe_obs = None
        #: the global novelty (fp64 [P]) and selection fitness F of this generation, this rank's rows of the novelty,
        #: the gathered characterisations [P, 3, 160] and the ids archived after the selection
        self.novelty = {r: None for r in ROLES}
        self.shaped_fitness = {r: None for r in ROLES}
        self._novelty_local = {r: None for r in ROLES}
        self._novelty_bc_all = None
        self.novelty_ids = {r: None for r in ROLES}
        if self.novelty_w or self.safe:
            # one tensor per role, shared by the novelty search and the safe mutations
            states = self.k.init_states(self.seed, NOVELTY_PROBE_TAG, _lib.NOVELTY_PROBES, self.device)
            self.novelty_probe_obs = {r: self.k.novelty_probe_obs(states, r) for r in ROLES}
        if self.novelty_w:
            self.novelty_ring = torch.zeros((len(ROLES), self.novelty_A, _lib.NOVELTY_BC_DIM), dtype=torch.float32,
                                            device=self.device)
            for i, r in enumerate(ROLES):          # slot 0: the founder the reference measures diversity against
                self.k.novelty_bc(self.founder[r].reshape(1, -1), layout.OBS_DIM[r], self.novelty_probe_obs[r],
                                  out=self.novelty_ring[i, 0:1], status=self.status)
            #: ring bookkeeping on the host (no sync needed): next slot to write, filled slots [0, filled), and the
            #: filled count this generation's novelty was measured against
            self.novelty_head, self.novelty_filled = 1 % self.novelty_A, 1
            self._novelty_eval_filled = None
        for r in ROLES:
            assert self.pop[r].shape[0] == self.shard.n_local, "population shard has the wrong row count"
        if int(args.elites_number) > self.P or int(args.elites_number) < 1:
            raise ValueError(f"elites_number must be in [1, population]: {args.elites_number} vs {self.P}")
        K_eff = 1 if (self.compat and not getattr(args, "play_discarded_hof_games", False)) else int(args.hof_size)
        self.variant = self.rollout_variant(self.P, K_eff)

    def _opponents(self, role):
        """Rows for the two other seats (ascending seat order), newest HoF entry
        first (``hof[len-1-k]``, genetic_algorithm.py:138-139,170-171,203-204)."""
        newest_first = {r: torch.flip(self.hof[r], dims=[0]).contiguous() for r in ROLES}
        if role == "agent_0":       # seats: adversary_0, agent_1
            return newest_first["adversary_0"], newest_first["agent_1"]
        if role == "agent_1":       # seats: adversary_0, agent_0
            return newest_first["adversary_0"], newest_first["agent_0"]
        # adversary: seats agent_0, agent_1; the reference seats hof_agent_0 in BOTH chairs
        # (genetic_algorithm.py:204, Appendix C #5)
        second = newest_first["agent_0"] if self.compat else newest_first["agent_1"]
        return newest_first["agent_0"], second

    def _rollout_spec(self, role, init):
        """(role, members, opp_a, opp_b, init) of one role's evaluation loop (genetic_algorithm.py:125-217)."""
        a = self.args
        K = int(a.hof_size)
        opp_a, opp_b = self._opponents(role)
        if self.compat and not getattr(a, "play_discarded_hof_games", False):
            # The reference plays hof_size games per member but OVERWRITES the reward each time
            # (`=`, genetic_algorithm.py:140,172,205; Appendix C #2): only the game against the
            # oldest HoF entry (k = K-1) reaches the fitness.  The discarded games are not
            # simulated here; their initial-state records are still drawn, so the game
            # that counts starts from the same state as in a reference run.
            opp_a, opp_b = opp_a[K - 1:K].contiguous(), opp_b[K - 1:K].contiguous()
            init = init[:, K - 1:K].contiguous()
        return (role, self.pop[role], opp_a, opp_b, init)

    def _finish_role(self, role, out):
        """Local rewards + distances of one role from its rollout results."""
        a = self.args
        K = int(a.hof_size)
        limit = a.max_timesteps_per_episode
        slot = self._role_slot(out, role, limit)                      # [n_local, K or 1, E]
        if self.compat:
            # only the LAST HoF game counts (reward overwritten, `=`), then / hof_size
            # (genetic_algorithm.py:140-144, Appendix C #2)
            reward = slot[:, -1, :].mean(dim=1) / K
        else:
            reward = slot.mean(dim=(1, 2))
        # fitness sharing against the frozen founder (Appendix C #3)
        dist_local = self.k.diversity_dist(self.pop[role], self.founder[role], layout.OBS_DIM[role])
        self._local[role] = (reward.contiguous(), dist_local)

    def _rollout_role(self, role, init):
        """Local rewards + distances of one role (genetic_algorithm.py:125-217)."""
        spec = self._rollout_spec(role, init)
        out = self._rollouts([spec], self.args.max_timesteps_per_episode)[role]
        self._finish_role(role, out)

    def evaluate(self):
        """The three evaluation loops -> global fitness fp64[P] per role; one fused all-gather."""
        a = self.args
        K = int(a.hof_size)
        # host-stream order of a reference run: role after role (genetic_algorithm.py:125-217)
        init = {r: self._initial_states(self.P, K, self.shard, ROLES.index(r) + 4 * self.gen) for r in ROLES}
        self._local = {}
        specs = [self._rollout_spec(r, init[r]) for r in ROLES]
        outs = self._rollouts(specs, a.max_timesteps_per_episode)
        for r in ROLES:
            self._finish_role(r, outs[r])
        if self.novelty_w:
            self._member_novelty()
        packed = torch.stack([torch.stack([self._local[r][0].to(torch.float64), self._local[r][1].to(torch.float64)]
                                          + ([self._novelty_local[r]] if self.novelty_w else []), dim=1)
                              for r in ROLES], dim=1)
        allp = self.comm.all_gather_rows(packed.contiguous(), self.shard)          # [P, 3, 2 or 3]
        for i, role in enumerate(ROLES):
            reward = allp[:, i, 0]
            div = self.k.diversity_from_dist(allp[:, i, 1].to(torch.float32))
            self.diversity[role] = div
            # applied regardless of --fitness_sharing in GA (Appendix C #4)
            if self.compat or a.fitness_sharing:
                reward = reward / (1.0 + div.to(reward.dtype))
            self.fitness[role] = reward.contiguous()
            if self.novelty_w:
                self.novelty[role] = allp[:, i, 2].contiguous()

    def _member_novelty(self):
        """Characterise this rank's members, gather the three roles' characterisations [P, 3, 160] in one
        all-gather, and measure each member's k-NN novelty against the other members and the role's archive."""
        bc = torch.empty((self.shard.n_local, len(ROLES), _lib.NOVELTY_BC_DIM), dtype=torch.float32,
                         device=self.device)
        for i, role in enumerate(ROLES):
            self.k.novelty_bc(self.pop[role], layout.OBS_DIM[role], self.novelty_probe_obs[role], out=bc[:, i],
                              status=self.status)
        self._novelty_bc_all = bc_all = self.comm.all_gather_rows(bc, self.shard)
        for i, role in enumerate(ROLES):
            self._novelty_local[role] = self.k.ga_novelty_knn(bc[:, i], self.shard.row0, bc_all[:, i],
                                                              self.novelty_ring[i], self.novelty_filled,
                                                              self.novelty_k)
        self._novelty_eval_filled = self.novelty_filled

    def _novelty_append(self):
        """Archive the characterisations of m members drawn on the device (the same ids on every rank, from the
        gathered characterisations: no collective), at ``head`` in draw order; the bookkeeping stays on the host."""
        h, m, A = self.novelty_head, self.novelty_m, self.novelty_A
        n1 = min(m, A - h)
        for i, role in enumerate(ROLES):
            ids = self.k.ga_novelty_draw(self.seed, self.gen, role, m, self.P, self.device)
            self.novelty_ids[role] = ids
            rows = self._novelty_bc_all[:, i].index_select(0, ids)                 # [m, 160]
            self.novelty_ring[i, h:h + n1] = rows[:n1]
            self.novelty_ring[i, :m - n1] = rows[n1:]
        self.novelty_head = (h + m) % A
        self.novelty_filled = min(self.novelty_filled + m, A)

    def evaluate_role(self, role):
        """Evaluation loop of one role alone (tests / tools) -> global fitness fp64[P]."""
        a = self.args
        init = self._initial_states(self.P, int(a.hof_size), self.shard, ROLES.index(role) + 4 * self.gen)
        self._local = {}
        self._rollout_role(role, init)
        reward, dist_local = self._local[role]
        dist_all = self.comm.all_gather_rows(dist_local, self.shard)
        div = self.k.diversity_from_dist(dist_all)
        self.diversity[role] = div
        if self.compat or a.fitness_sharing:
            reward = reward / (1.0 + div.to(reward.dtype))
        self.fitness[role] = self.comm.all_gather_rows(reward.contiguous(), self.shard)
        return self.fitness[role]

    def select_and_repopulate(self):
        """Truncation selection, HoF FIFO update, elite cloning + mutation
        (genetic_algorithm.py:223-290) for the three roles; the elite indices never leave the
        device and the three roles' elite rows travel in ONE all-reduce."""
        a = self.args
        E = int(a.elites_number)
        # with novelty search one more row per role: the fitness-best member, for the HoF and the evaluation games
        rows = E + 1 if self.novelty_w else E
        pitches = [layout.fc_pitch(layout.OBS_DIM[r]) for r in ROLES]
        cat = torch.empty(rows * sum(pitches), dtype=torch.float32, device=self.device)
        views, off = {}, 0
        for r, pitch in zip(ROLES, pitches):
            views[r] = cat[off:off + rows * pitch].view(rows, pitch)
            off += rows * pitch
        if self.novelty_w:
            # each rank ranks its own rows; F is combined in fp64 and gathered for the three roles at once
            w = self.novelty_w
            F_local = torch.stack([(1.0 - w) * self.k.centered_ranks(self.fitness[r], self.shard.row0,
                                                                     self.shard.n_local)
                                   + w * self.k.centered_ranks(self.novelty[r], self.shard.row0, self.shard.n_local)
                                   for r in ROLES], dim=1)
            F_all = self.comm.all_gather_rows(F_local.contiguous(), self.shard)      # [P, 3]
        for i, role in enumerate(ROLES):
            if self.novelty_w:
                self.shaped_fitness[role] = F_all[:, i].contiguous()
                ids = self.k.select_topk(self.shaped_fitness[role], E, order=self.order)
                best = self.k.select_topk(self.fitness[role], 1, order=self.order)
                self.elite_ids[role] = ids
                ids = torch.cat([ids, best])
            else:
                ids = self.k.select_topk(self.fitness[role], E, order=self.order)    # replicated, bit-exact
                self.elite_ids[role] = ids
            # owner rows, zeros elsewhere; summed over ranks = the elite / HoF broadcast
            self.k.gather_rows(self.pop[role], ids, row0=self.shard.row0, n_local=self.shard.n_local,
                               out=views[role])
        self.comm.all_reduce_sum(cat)
        for role in ROLES:
            in_dim = layout.OBS_DIM[role]
            elites = views[role][:E] if self.novelty_w else views[role]
            self.elites[role] = elites
            best = views[role][E:E + 1] if self.novelty_w else elites[0:1]
            self.best_rows[role] = best[0]
            # HoF: append the best, drop the oldest (genetic_algorithm.py:270-275)
            self.hof[role] = torch.cat([self.hof[role][1:], best], dim=0).contiguous()
            # next population: row 0 = best unmutated, rows c>=1 = elites[(c-1)%E] + sigma*N(0,1)
            # (with safe mutations: + fl(sigma*N(0,1)) * c, c the scale row of the elite)
            extra = {}
            if self.safe:
                self.safe_scale[role] = extra["scale"] = self.k.ga_safe_scale(
                    elites, in_dim, self.novelty_probe_obs[role], self.safe_floor, status=self.status)
            self.k.ga_repopulate(elites, layout.fc_dim(in_dim), self.sigma_dev(role), self.seed, role, self.gen,
                                 self.shard.row0, self.shard.n_local, out=self.pop[role],
                                 crossover_rate=float(getattr(a, "crossover_rate", 0.0)), **extra)
        if self.novelty_w:
            self._novelty_append()

    def step(self, sync=True):
        """One generation.  ``sync=True`` returns the evaluation triple (one host read);
        ``sync=False`` issues the generation without a host round trip."""
        self._raise_pending_status()
        if self.adaptive:
            self._join_eval()             # this generation's sigma is the previous generation's output
        self.evaluate()
        self.select_and_repopulate()
        best = self.best_rows
        self._finish_generation(best["agent_0"], best["agent_1"], best["adversary_0"])
        if self.history is not None:
            hs = self.host_state()
            self.check_status()
            nov = self.novelty_w

            def host(t):
                return {r: t[r].cpu().numpy().copy() for r in ROLES} if nov else None
            self.history.append(dict(
                fitness={r: self.fitness[r].cpu().numpy().copy() for r in ROLES},
                elite_ids={r: self.elite_ids[r].cpu().numpy().copy() for r in ROLES},
                diversity={r: float(self.diversity[r]) for r in ROLES}, evals=self.last_eval(),
                sigma={r: float(hs["sigma_history"][r][self.gen]) for r in ROLES},
                novelty=host(self.novelty), novelty_filled=self._novelty_eval_filled if nov else None,
                shaped_fitness=host(self.shaped_fitness), novelty_archive_ids=host(self.novelty_ids),
                safe_mutation_scale=self._safe_scale_stats() if self.safe else None))
        self.gen += 1
        return self.last_eval() if sync else None

    def _safe_scale_stats(self):
        """Per role the mean, min and max of this generation's scales c over the E x D entries of the elites, and the
        count of entries at 1 / floor (reduced on the device, one host read)."""
        at_floor = np.float32(1.0) / np.float32(self.safe_floor)
        stats = []
        for r in ROLES:
            c = self.safe_scale[r][:, :layout.fc_dim(layout.OBS_DIM[r])]
            stats.append(torch.stack([c.mean(dtype=torch.float64), c.min().double(), c.max().double(),
                                      (c == float(at_floor)).sum().double()]))
        host = torch.stack(stats).cpu().numpy()
        return {r: dict(mean=float(v[0]), min=float(v[1]), max=float(v[2]), n_floor=int(v[3]))
                for r, v in zip(ROLES, host)}

    def state_dict(self):
        """Everything a run needs to continue bit for bit: this rank's population shard, the HoF
        ring, founders, generation state (sigmas, histories, counters), the host init-state stream, and the
        novelty-search settings, with novelty search its characterisation rings and their bookkeeping (the probe
        observations are a function of the seed)."""
        sd = self._base_state()
        sd.update(pop={r: self.pop[r].cpu() for r in ROLES}, hof={r: self.hof[r].cpu() for r in ROLES},
                  founder={r: self.founder[r].cpu() for r in ROLES}, ga_novelty=dict(self.novelty_opts),
                  ga_safe_mutation=dict(self.safe_opts))
        if self.novelty_w:
            sd.update(novelty_ring=self.novelty_ring.cpu().clone(), novelty_head=self.novelty_head,
                      novelty_filled=self.novelty_filled)
        return sd

    def load_state_dict(self, sd):
        """Refuses a checkpoint written with other novelty-search or safe-mutation settings (one without them was
        written with the option off)."""
        saved = sd.get("ga_novelty", GA_NOVELTY_DEFAULTS)
        if saved != self.novelty_opts:
            raise ValueError(f"checkpoint was written with the GA novelty search {saved}, this run uses "
                             f"{self.novelty_opts}")
        saved = sd.get("ga_safe_mutation", GA_SAFE_MUTATION_DEFAULTS)
        if saved != self.safe_opts:
            raise ValueError(f"checkpoint was written with the GA safe mutations {saved}, this run uses "
                             f"{self.safe_opts}")
        self._load_base_state(sd)
        if int(sd["row0"]) != self.shard.row0 or int(sd["n_local"]) != self.shard.n_local:
            raise ValueError("checkpoint shard does not match this rank's row block (same world size needed)")
        for r in ROLES:
            self.pop[r].copy_(sd["pop"][r])
            self.hof[r] = sd["hof"][r].to(self.device).contiguous()
            self.founder[r].copy_(sd["founder"][r])
        if self.novelty_w:
            self.novelty_ring.copy_(sd["novelty_ring"])
            self.novelty_head, self.novelty_filled = int(sd["novelty_head"]), int(sd["novelty_filled"])


# ---------------------------------------------------------------------------
# Co-ES  (evolutionary_strategy.py:151-393)
# ---------------------------------------------------------------------------
class ESEngine(_EngineBase):
    """State: one replicated base row per role.  Members of a generation are
    ``theta + sigma * N(0,1)`` regenerated from the Philox key both when they are
    materialised for the rollout (K5) and when the update is formed (K6).

    Opt-in update options (``es_options``): mirrored sampling (members 2q and 2q+1 are
    ``theta +- sigma * z_q``), centered-rank fitness shaping of the global fitness, and an Adam step
    and / or L2 weight decay applied by one fused kernel after the delta all-reduce (K6 then yields
    the ascent estimate itself, at lr = 1).  Adam's moments ``m`` / ``v`` are laid out like
    ``theta_cat`` and replicated like it.

    Opt-in search distribution (``es_distribution``): separable NES keeps a per-parameter sigma
    (``sigma_cat``, laid out like ``theta_cat`` and replicated like it) that the population's rewards adapt
    through the natural gradient of log sigma; K5 / K6 / the apply become their diag forms.

    Opt-in Hall of Fame (``es_hof``): an archive ring ``hof_ring`` fp32 [H, len(theta_cat)] of ``theta_cat``
    snapshots (the founders, then one after every apply), replicated like theta.  Every member then plays K
    opponent sets of E games each: set 0 is the current base agents, sets 1..K-1 are snapshots drawn on the device
    (``cev_es_hof_opponents_i64``, keyed by (seed, generation)), and its reward is the mean over the K x E games.

    Opt-in guided search (``es_subspace``): a ring ``subspace_ring`` fp32 [k, len(theta_cat)] of the last k all-reduced
    update estimates (``delta_cat``), replicated like theta, and its orthonormal basis ``subspace_U`` (k_eff <= k rows
    per role, ``cev_es_subspace_basis_f32``, recomputed after every apply).  Members are theta + sigma (A z + B U^T c):
    a share alpha of the variance stays isotropic, the rest lies in the subspace, with the total variance of the
    isotropic search.  The update is the default members-form K6, which reads sigma eps back as member - theta.

    Opt-in novelty search (``es_novelty``, NS-ES / NSR-ES): a member's behaviour characterisation is its softmax action
    distributions on 32 probe observations (``novelty_probe_obs``, drawn once from the seed), fp32 [160].  Per role a
    ring ``novelty_ring`` fp32 [A, 160] holds those of past base agents (the founders, then one after every apply),
    replicated like theta; a member's novelty is the mean distance to its k nearest entries, and the update is
    weighted by F = (1 - w) cr(reward) + w cr(novelty) (cr: centered ranks of the global vectors).

    Opt-in LM-MA-ES (``es_distribution`` 'lmma', Loshchilov et al. 2019): m direction vectors per role ``lmma_M`` fp32
    [m, len(theta_cat)], the path ``lmma_p`` and the Gram ``lmma_G`` fp64 [3, m, m], replicated like theta.  Members are
    theta + sigma (alpha z + sum_l beta_l m_l) through the first k = min(g, m) vectors; the mu best are recombined with
    log weights, and the apply steps theta, the path, the vectors and sigma (cumulative step-size adaptation)."""

    kind = "ES"
    #: Philox stream of the initial states of ``hof_matrix``
    _hof_matrix_tag = 0x50000000

    def __init__(self, args, device, theta_rows, env=None, kernels=None, comm=None):
        super().__init__(args, device, env, kernels, comm)
        self.P = int(args.population)
        self.options = es_options(args, "ES")
        ga_novelty(args, "ES")                           # refuses the Co-GA options
        ga_safe_mutation(args, "ES")
        self.mirrored = self.options["mirrored_sampling"]
        self.shaping = self.options["fitness_shaping"] == "centered_rank"
        #: the fused apply kernel instead of K6 at lr + axpy (the default path)
        self.fused_apply = self.options["es_optimizer"] == "adam" or self.options["l2_coeff"] != 0.0
        self.shard = Shard(self.P, self.comm.rank, self.comm.world)
        pitches = [layout.fc_pitch(layout.OBS_DIM[r]) for r in ROLES]
        # the three base rows / deltas live in one buffer each: one all-reduce, one apply
        self.theta_cat = torch.empty(sum(pitches), dtype=torch.float32, device=self.device)
        self.delta_cat = torch.zeros(sum(pitches), dtype=torch.float32, device=self.device)
        self.theta, self.last_delta, off = {}, {}, 0
        for r, pitch in zip(ROLES, pitches):
            self.theta[r] = self.theta_cat[off:off + pitch]
            self.last_delta[r] = self.delta_cat[off:off + pitch]
            self.theta[r].copy_(theta_rows[r].reshape(-1)[:pitch])
            off += pitch
        self.comm.broadcast0(self.theta_cat)              # rank 0's base agents everywhere (ADVICE r1)
        #: (offset, pitch) of each role's row in theta_cat (every offset is a multiple of 32 floats)
        self.cols = {r: (o, p) for r, o, p in zip(ROLES, np.cumsum([0] + pitches[:-1]).tolist(), pitches)}
        self.hof_opts = es_hof(args, "ES")
        self.hof_size = self.hof_opts["es_hof_size"]
        #: opponent sets per member: K with the Hall of Fame, else the current base agents only
        self.K = self.hof_opts["es_hof_opponents"] if self.hof_size else 1
        self.hof_ring = self.hof_opp = self.hof_ids = None
        if self.hof_size:
            n = self.theta_cat.numel()
            self.hof_ring = torch.zeros((self.hof_size, n), dtype=torch.float32, device=self.device)
            self.hof_ring[0].copy_(self.theta_cat)
            #: ring bookkeeping on the host (no sync needed): next slot to write, filled slots [0, filled), and
            #: the generation whose base agents each slot holds (-1: empty)
            self.hof_head, self.hof_filled = 1 % self.hof_size, 1
            self.hof_slot_gen = [0] + [-1] * (self.hof_size - 1)
            #: this generation's K snapshots, gathered once: the roles' opponents are column views of it
            self.hof_opp = torch.empty((self.K, n), dtype=torch.float32, device=self.device)
            self.hof_ids = torch.empty(self.K, dtype=torch.int64, device=self.device)
            self._hof_eval_slot_gen = None
        self.distribution = es_distribution(args, "ES")
        self.separable = self.distribution["es_distribution"] == "separable"
        #: LM-MA-ES: m direction vectors per role (0: off)
        self.lmma_m = self.distribution.get("es_lmma_memory", 0)
        self.subspace_opts = es_subspace(args, "ES")
        #: guided-search subspace dimension k (0: off) and the share alpha of the variance outside it
        self.subspace_k = self.subspace_opts["es_subspace_dim"]
        self.subspace_alpha = self.subspace_opts["es_subspace_alpha"]
        self.subspace_ring = self.subspace_U = self.subspace_keff = None
        if self.subspace_k:
            n = self.theta_cat.numel()
            self.subspace_ring = torch.zeros((self.subspace_k, n), dtype=torch.float32, device=self.device)
            self.subspace_U = torch.zeros((self.subspace_k, n), dtype=torch.float32, device=self.device)
            #: k_eff per role on the device (K5 reads it there): 0 until the first estimate
            self.subspace_keff = torch.zeros(len(ROLES), dtype=torch.int32, device=self.device)
            #: ring bookkeeping on the host (no sync needed): next slot to write, filled slots [0, filled)
            self.subspace_head, self.subspace_filled = 0, 0
        self.novelty_opts = es_novelty(args, "ES")
        #: novelty weight w (0: off), nearest neighbours k and archive capacity A
        self.novelty_w = self.novelty_opts["es_novelty_weight"]
        self.novelty_k = self.novelty_opts["es_novelty_k"]
        self.novelty_A = self.novelty_opts["es_novelty_archive"]
        self.novelty_ring = self.novelty_probe_obs = None
        #: the global novelty of this generation's members (fp64 [P] per role) and this rank's rows of it
        self.novelty = {r: None for r in ROLES}
        self._novelty_local = {r: None for r in ROLES}
        if self.novelty_w:
            states = self.k.init_states(self.seed, NOVELTY_PROBE_TAG, _lib.NOVELTY_PROBES, self.device)
            self.novelty_probe_obs = {r: self.k.novelty_probe_obs(states, r) for r in ROLES}
            self.novelty_ring = torch.zeros((len(ROLES), self.novelty_A, _lib.NOVELTY_BC_DIM), dtype=torch.float32,
                                            device=self.device)
            #: ring bookkeeping on the host (no sync needed): next slot to write, filled slots [0, filled), and the
            #: filled count this generation's novelty was measured against
            self.novelty_head, self.novelty_filled = 0, 0
            self._novelty_eval_filled = None
            self._novelty_append()
        self.sigma_cat = self.grad_cat = None
        self.sigma_rows, self.sigma_grad, self.sigma_lr = {}, {}, {}
        if self.separable:
            # per-parameter sigma laid out like theta_cat (sigma0 on the Linear entries, 0 elsewhere), replicated like
            # it; grad_cat = [g_mu of the roles | g_sigma of the roles]: still one all-reduce per generation
            n = self.theta_cat.numel()
            self.sigma_cat = torch.zeros(n, dtype=torch.float32, device=self.device)
            self.grad_cat = torch.zeros(2 * n, dtype=torch.float32, device=self.device)
            self.delta_cat = self.grad_cat[:n]
            sigma0 = {"agent_0": args.mutation_power_agent_0, "agent_1": args.mutation_power_agent_1,
                      "adversary_0": args.mutation_power_adversary}
            off = 0
            for r, pitch in zip(ROLES, pitches):
                pidx = torch.from_numpy(layout.fc_perturbable_index(layout.OBS_DIM[r]))
                row = torch.zeros(pitch, dtype=torch.float32)
                row[pidx] = float(np.float32(sigma0[r]))
                self.sigma_rows[r] = self.sigma_cat[off:off + pitch]
                self.sigma_rows[r].copy_(row)
                self.last_delta[r] = self.grad_cat[off:off + pitch]
                self.sigma_grad[r] = self.grad_cat[n + off:n + off + pitch]
                lr = self.distribution["sigma_learning_rate"]
                self.sigma_lr[r] = float(lr) if lr is not None else default_sigma_learning_rate(len(pidx))
                off += pitch
        self.lmma_M = self.lmma_p = self.lmma_G = None
        if self.lmma_m:
            self._lmma_init(pitches)
        self.adam_m = self.adam_v = None
        if self.options["es_optimizer"] == "adam":
            self.adam_m = torch.zeros_like(self.theta_cat)
            self.adam_v = torch.zeros_like(self.theta_cat)
        self.members = {r: torch.empty((self.shard.n_local, layout.fc_pitch(layout.OBS_DIM[r])),
                                       dtype=torch.float32, device=self.device) for r in ROLES}
        self.fitness = {r: None for r in ROLES}
        #: this rank's rows of the centered-rank shaped fitness the update used (fitness shaping only)
        self.shaped_fitness = {r: None for r in ROLES}
        self.rewards = {r: None for r in ROLES}
        self.diversity = {r: None for r in ROLES}
        self.weight_stats = {r: None for r in ROLES}      # fp32 [n_local, 4] when args.log_member_weight_stats
        self.member_stats = bool(getattr(args, "log_member_weight_stats", False))
        self.variant = self.rollout_variant(self.P, self.K)

    def _lmma_init(self, pitches):
        """LM-MA-ES state, replicated like theta: the direction vectors M fp32 [m, len(theta_cat)] (zero), the path p
        fp32 [len(theta_cat)] (zero), the Gram of each role's vectors fp64 [3, m, m] and the update count g; and
        grad_cat = [zbar of the roles | betabar fp32 [3, m]], so a generation still has one all-reduce."""
        m, n = self.lmma_m, self.theta_cat.numel()
        self.lmma_M = torch.zeros((m, n), dtype=torch.float32, device=self.device)
        self.lmma_p = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.lmma_G = torch.zeros((len(ROLES), m, m), dtype=torch.float64, device=self.device)
        self.lmma_stats = torch.zeros((len(ROLES), 2), dtype=torch.float64, device=self.device)
        self.lmma_gen = 0
        self.grad_cat = torch.zeros(n + len(ROLES) * m, dtype=torch.float32, device=self.device)
        self.delta_cat = self.grad_cat[:n]
        self.lmma_betabar = self.grad_cat[n:].view(len(ROLES), m)
        off = 0
        for r, pitch in zip(ROLES, pitches):
            self.last_delta[r] = self.grad_cat[off:off + pitch]
            off += pitch
        #: per role: the constants (n = the role's Linear entries), the weights on the device, this generation's
        #: transform coefficients beta fp32 [n_local, k] and selected ids
        self.lmma_const = {r: lmma_constants(self.P, len(layout.fc_perturbable_index(layout.OBS_DIM[r])), m)
                           for r in ROLES}
        self.lmma_w = {r: torch.tensor(c["w"], dtype=torch.float32).to(self.device) for r, c in self.lmma_const.items()}
        self.lmma_beta = {r: None for r in ROLES}
        self.lmma_ids = {r: None for r in ROLES}

    def _lmma_k(self):
        """Vectors in use this generation: k = min(g, m)."""
        return min(self.lmma_gen, self.lmma_m)

    def _lmma_perturb(self, role):
        """K5 of LM-MA-ES: the isotropic K5 while k = 0, else the projection and the LM-MA K5."""
        in_dim, k = layout.OBS_DIM[role], self._lmma_k()
        if k == 0:
            self.lmma_beta[role] = torch.zeros((self.shard.n_local, 0), dtype=torch.float32, device=self.device)
            self.k.es_perturb(self.theta[role], in_dim, self.sigma_dev(role), self.seed, role, self.gen,
                              self.shard.row0, self.shard.n_local, out=self.members[role])
            return
        o, p = self.cols[role]
        c = self.lmma_const[role]
        M = self.lmma_M[:, o:o + p]
        beta = self.k.es_lmma_project(M, k, self.lmma_G[ROLES.index(role)], c["c_d"][:k], in_dim, self.seed, role,
                                      self.gen, self.shard.row0, self.shard.n_local, status=self.status)
        self.lmma_beta[role] = beta
        self.k.es_perturb_lmma(self.theta[role], in_dim, self.sigma_dev(role), M, k, beta, c["alpha"][k], self.seed,
                               role, self.gen, self.shard.row0, self.shard.n_local, out=self.members[role])

    def _lmma_update(self):
        """Select the mu best of the global fitness (ties to the lower index, NaN last, whatever reference_compat
        says: the reference has no LM-MA-ES), recombine this rank's selected normals, all-reduce, apply."""
        a = self.args
        k = self._lmma_k()
        for i, role in enumerate(ROLES):
            c = self.lmma_const[role]
            ids = self.k.select_topk(self.fitness[role], c["mu"], order=_lib.ORDER_STABLE_DESC)
            self.lmma_ids[role] = ids
            self.k.es_lmma_reduce(ids, self.lmma_w[role], self.lmma_beta[role], layout.OBS_DIM[role], self.seed, role,
                                  self.gen, self.shard.row0, self.shard.n_local, zbar=self.last_delta[role],
                                  betabar=self.lmma_betabar[i, :k])
        self.comm.all_reduce_sum(self.grad_cat)
        self._join_eval()                 # the previous generation's evaluation games read theta and sigma
        # replicated on every rank from the same all-reduced buffer: the replicas stay identical
        cs = [self.lmma_const[r] for r in ROLES]
        self.k.es_lmma_apply(self.theta_cat, self.lmma_M, self.lmma_p, self.delta_cat, self.lmma_betabar,
                             [layout.OBS_DIM[r] for r in ROLES], k=k, alpha=[c["alpha"][k] for c in cs],
                             c_sigma=[c["c_sigma"] for c in cs], mu_w=[c["mu_w"] for c in cs], c_m=a.learning_rate,
                             c_c=[c["c_c"] for c in cs], G=self.lmma_G, gstate=self.gstate,
                             sigma_min=a.min_mutation_power, sigma_max=a.max_mutation_power, stats=self.lmma_stats,
                             status=self.status)
        self.lmma_gen += 1

    def _lmma_record(self, k):
        """History record of LM-MA-ES: per role the vectors used, |p_sigma|^2 / n and sigma after the update."""
        st = self.lmma_stats.cpu().numpy()
        return {r: {"k_eff": k, "p_sigma_norm2_over_n": float(st[i, 0]), "sigma_after": float(st[i, 1])}
                for i, r in enumerate(ROLES)}

    def _base_opponents(self, role):
        """Rows of the two other seats (ascending seat order): the base rows [1, pitch], or with the Hall of Fame the
        roles' columns of this generation's K gathered snapshots [K, pitch] (row pitch len(theta_cat))."""
        if self.hof_size:
            t = {r: self.hof_opp[:, o:o + p] for r, (o, p) in self.cols.items()}
        else:
            t = {r: self.theta[r].reshape(1, -1) for r in ROLES}
        if role == "agent_0":
            return t["adversary_0"], t["agent_1"]
        if role == "agent_1":
            return t["adversary_0"], t["agent_0"]
        return t["agent_0"], t["agent_1"]

    def _reference_initial_states(self):
        """The reference interleaves the three roles per member
        (evolutionary_strategy.py:236-251): game 3*i + role_index; with K opponent sets the
        records of a member and role are laid out [K, E]."""
        K, E = self.K, self.E
        block = self.env.draw_initial_states(self.P * 3 * K * E).reshape(self.P, 3, K, E, mpe_spec.INIT_STATE_DIM)
        sl = slice(self.shard.row0, self.shard.row0 + self.shard.n_local)
        return {r: torch.from_numpy(np.ascontiguousarray(block[sl, i])).to(self.device)
                for i, r in enumerate(ROLES)}

    def _gather_hof_opponents(self):
        """The K opponent snapshots of this generation: slots drawn on the device, rows gathered from the ring."""
        newest = (self.hof_head - 1) % self.hof_size
        self.k.es_hof_opponents(self.seed, self.gen, self.K, self.hof_filled, newest, self.device, out=self.hof_ids)
        self.k.gather_rows(self.hof_ring, self.hof_ids, out=self.hof_opp)
        self._hof_eval_slot_gen = list(self.hof_slot_gen)

    def _hof_append(self):
        """Archive the base agents just applied (a stream-ordered device copy; the bookkeeping stays on the host)."""
        self.hof_ring[self.hof_head].copy_(self.theta_cat)
        self.hof_slot_gen[self.hof_head] = self.gen + 1
        self.hof_head = (self.hof_head + 1) % self.hof_size
        self.hof_filled = min(self.hof_filled + 1, self.hof_size)

    def evaluate(self, init_by_role=None):
        """Perturb + one rollout per member and role against the other roles'
        BASE policies (mutate_weights, evolutionary_strategy.py:63-116), or with the
        Hall of Fame against K opponent sets.
        ``init_by_role`` (optional) supplies the initial states [n_local,K,E,11] per role."""
        limit = self.args.max_timesteps_per_episode
        ref_init = init_by_role
        if ref_init is None and self.init_mode == "reference":
            ref_init = self._reference_initial_states()
        if self.hof_size:
            self._gather_hof_opponents()

        specs = {}

        def prepare(role):
            in_dim = layout.OBS_DIM[role]
            if self.separable:
                self.k.es_perturb_diag(self.theta[role], self.sigma_rows[role], in_dim, self.seed, role, self.gen,
                                       self.shard.row0, self.shard.n_local, mirrored=self.mirrored,
                                       out=self.members[role])
            elif self.lmma_m:
                self._lmma_perturb(role)
            elif self.subspace_k:
                o, p = self.cols[role]
                i = ROLES.index(role)
                self.k.es_perturb_subspace(self.theta[role], in_dim, self.sigma_dev(role), self.subspace_U[:, o:o + p],
                                           self.subspace_keff[i:i + 1], self.subspace_alpha, self.seed, role, self.gen,
                                           self.shard.row0, self.shard.n_local, mirrored=self.mirrored,
                                           out=self.members[role])
            else:
                perturb = self.k.es_perturb_mirrored if self.mirrored else self.k.es_perturb
                perturb(self.theta[role], in_dim, self.sigma_dev(role), self.seed, role, self.gen,
                        self.shard.row0, self.shard.n_local, out=self.members[role])
            if self.member_stats:
                # per-member statistics of the perturbed weights (MPE/mpe_agent.py:30-50, agent.py:66)
                self.weight_stats[role] = self.k.weight_stats(self.members[role], in_dim)
            if ref_init is not None:
                init = ref_init[role]
            else:
                init = self._initial_states(self.P, self.K, self.shard, ROLES.index(role) + 4 * self.gen)
            opp_a, opp_b = self._base_opponents(role)
            specs[role] = (role, self.members[role], opp_a, opp_b, init)

        self._run_roles(prepare)
        outs = self._rollouts([specs[r] for r in ROLES], limit)
        for role in ROLES:
            slot = self._role_slot(outs[role], role, limit)           # [n_local, K, E]
            self.rewards[role] = slot.mean(dim=(1, 2)).contiguous()   # the mean over all K x E games
        if self.novelty_w:
            self._member_novelty()

    def _member_novelty(self):
        """Behaviour characterisations of this rank's members and their k-NN novelty against the role's archive."""
        for i, role in enumerate(ROLES):
            bc = self.k.novelty_bc(self.members[role], layout.OBS_DIM[role], self.novelty_probe_obs[role],
                                   status=self.status)
            self._novelty_local[role] = self.k.novelty_knn(bc, self.novelty_ring[i], self.novelty_filled, self.novelty_k)
        self._novelty_eval_filled = self.novelty_filled

    def _novelty_append(self):
        """Characterise the current base agents straight into slot ``head`` of each role's ring (bookkeeping on the
        host)."""
        h = self.novelty_head
        for i, role in enumerate(ROLES):
            self.k.novelty_bc(self.theta[role].reshape(1, -1), layout.OBS_DIM[role], self.novelty_probe_obs[role],
                              out=self.novelty_ring[i, h:h + 1], status=self.status)
        self.novelty_head = (h + 1) % self.novelty_A
        self.novelty_filled = min(self.novelty_filled + 1, self.novelty_A)

    def update(self):
        """compute_weight_update + apply (evolutionary_strategy.py:120-148,255-265) for the three
        roles: one fitness all-gather, three K6 launches into one buffer, one all-reduce, one apply."""
        a = self.args
        # the reference casts rewards to fp32 before the update (np.array(rewards, dtype=np_dtype))
        fit_local = {r: self.rewards[r].to(torch.float32).to(torch.float64) for r in ROLES}
        cols = [fit_local[r] for r in ROLES]
        if a.fitness_sharing:
            cols += [self.k.diversity_dist(self.members[r], self.theta[r], layout.OBS_DIM[r]).to(torch.float64)
                     for r in ROLES]
        nov0 = len(cols)                  # the novelty columns, when on
        if self.novelty_w:
            cols += [self._novelty_local[r] for r in ROLES]
        packed = torch.stack(cols, dim=1).contiguous()                             # [n_local, 3, 6 or 9]
        start = getattr(self.comm, "all_gather_rows_start", None)                  # injected comms may only gather
        if start is not None:
            gathered = start(packed, self.shard)                                   # -> [P, 3 or 6]
        else:
            _all = self.comm.all_gather_rows(packed, self.shard)
            gathered = lambda: _all

        def finish_fitness():
            allp = gathered()
            for i, role in enumerate(ROLES):
                if a.fitness_sharing:
                    div = self.k.diversity_from_dist(allp[:, 3 + i].to(torch.float32))
                    self.diversity[role] = div
                    fit_local[role] = (fit_local[role].to(torch.float32) / (1 + div)).to(torch.float64)
                    self.fitness[role] = (allp[:, i].to(torch.float32) / (1 + div)).to(torch.float64)
                else:
                    self.fitness[role] = allp[:, i].contiguous()
                if self.novelty_w:
                    self.novelty[role] = allp[:, nov0 + i].contiguous()

        if self.lmma_m:
            finish_fitness()              # the selection ranks the global fitness
            self._lmma_update()
            if self.hof_size:
                self._hof_append()
            return
        need_global = a.fitness_sharing or self.shaping
        if need_global:
            finish_fitness()              # the update needs the shared fitness / the ranks of the global fitness
        # with the fused apply K6 yields the ascent estimate ghat (lr = 1); the step size is applied after it
        lr = 1.0 if self.fused_apply else a.learning_rate
        for role in ROLES:
            in_dim = layout.OBS_DIM[role]
            fit = fit_local[role].contiguous()
            if self.shaping:
                # ranks over the global fitness (after sharing: its division by one positive scalar keeps the order)
                fit = self.k.centered_ranks(self.fitness[role], self.shard.row0, self.shard.n_local)
                if self.novelty_w:
                    # NSR-ES (NS-ES at w = 1): the ranks of the reward and of the novelty, combined in fp64
                    w = self.novelty_w
                    fit = (1.0 - w) * fit + w * self.k.centered_ranks(self.novelty[role], self.shard.row0,
                                                                      self.shard.n_local)
                self.shaped_fitness[role] = fit
            if self.separable:
                # always from regenerated noise: z = (member - theta) / sigma would not be exact
                self.k.es_update_diag(fit, in_dim, self.P, self.seed, role, self.gen, self.shard.row0,
                                      mirrored=self.mirrored, g_mu=self.last_delta[role], g_sigma=self.sigma_grad[role])
            elif self.update_from_members and hasattr(self.k, "es_update_members"):
                # sigma*z_i read back from the materialised members (HBM bound) instead of regenerated
                self.k.es_update_members(fit, self.members[role], self.theta[role],
                                         in_dim, self.sigma_dev(role), lr, self.P,
                                         out=self.last_delta[role])
            else:
                update = self.k.es_update_mirrored if self.mirrored else self.k.es_update
                update(fit, in_dim, self.sigma_dev(role), lr,
                       self.P, self.seed, role, self.gen, self.shard.row0, out=self.last_delta[role])
        if not need_global:
            finish_fitness()              # the global fitness is a record only: gathered under the three K6 launches
        self.comm.all_reduce_sum(self.grad_cat if self.separable else self.delta_cat)
        self._join_eval()                 # the previous generation's evaluation games read theta
        if self.separable:
            # replicated on every rank from the same all-reduced gradients: the replicas stay identical
            n = self.theta_cat.numel()
            self.k.es_apply_diag(self.theta_cat, self.sigma_cat, self.grad_cat[:n], self.grad_cat[n:],
                                 [layout.OBS_DIM[r] for r in ROLES], lr=a.learning_rate,
                                 sigma_lr=[self.sigma_lr[r] for r in ROLES], sigma_min=a.min_mutation_power,
                                 sigma_max=a.max_mutation_power)
        elif self.fused_apply:
            # replicated on every rank from the same all-reduced delta: the replicas stay identical
            self.k.es_apply(self.theta_cat, self.delta_cat, [layout.OBS_DIM[r] for r in ROLES],
                            optimizer=self.options["es_optimizer"], lr=a.learning_rate,
                            l2_coeff=self.options["l2_coeff"], t=self.gen + 1, m=self.adam_m, v=self.adam_v)
        else:
            self.k.axpy(1.0, self.delta_cat, self.theta_cat)
        if self.hof_size:
            self._hof_append()
        if self.subspace_k:
            self._subspace_append()
        if self.novelty_w:
            self._novelty_append()

    def _subspace_append(self):
        """Append this generation's all-reduced estimate to the ring (a stream-ordered device copy; the bookkeeping
        stays on the host) and recompute the basis on the device."""
        self.subspace_ring[self.subspace_head].copy_(self.delta_cat)
        self.subspace_head = (self.subspace_head + 1) % self.subspace_k
        self.subspace_filled = min(self.subspace_filled + 1, self.subspace_k)
        self._subspace_basis()

    def _subspace_basis(self):
        newest = (self.subspace_head - 1) % self.subspace_k
        self.k.es_subspace_basis(self.subspace_ring, newest, self.subspace_filled, [layout.OBS_DIM[r] for r in ROLES],
                                 out=self.subspace_U, k_eff=self.subspace_keff)

    def step(self, init_by_role=None, sync=True):
        """One generation.  ``sync=True`` returns the evaluation triple (one host read);
        ``sync=False`` issues the generation without a host round trip."""
        self._raise_pending_status()
        if self.adaptive:
            self._join_eval()             # this generation's sigma is the previous generation's output
        lmma_k = self._lmma_k() if self.lmma_m else None
        self.evaluate(init_by_role)
        self.update()
        self._finish_generation(self.theta["agent_0"], self.theta["agent_1"], self.theta["adversary_0"])
        if self.history is not None:
            hs = self.host_state()
            self.check_status()
            rewards_all = {r: self.comm.all_gather_rows(self.rewards[r], self.shard).cpu().numpy().copy()
                           for r in ROLES}
            self.history.append(dict(
                rewards=rewards_all,
                diversity={r: (float(self.diversity[r]) if self.diversity[r] is not None else None) for r in ROLES},
                evals=self.last_eval(),
                delta={r: self.last_delta[r].cpu().numpy().copy() for r in ROLES},
                shaped_fitness={r: (self.comm.all_gather_rows(self.shaped_fitness[r], self.shard).cpu().numpy().copy()
                                    if self.shaping else None) for r in ROLES},
                sigma={r: float(hs["sigma_history"][r][self.gen]) for r in ROLES},
                sigma_stats={r: self._sigma_stats(r) for r in ROLES},
                hof_ids=self._hof_ids_record(),
                subspace_rank=({r: int(x) for r, x in zip(ROLES, self.subspace_keff.cpu().tolist())}
                               if self.subspace_k else None),
                novelty=({r: self.novelty[r].cpu().numpy().copy() for r in ROLES} if self.novelty_w else None),
                novelty_filled=self._novelty_eval_filled if self.novelty_w else None,
                lmma=self._lmma_record(lmma_k) if self.lmma_m else None))
        self.gen += 1
        return self.last_eval() if sync else None

    def _hof_ids_record(self):
        """(archive slots, their generations) of this generation's K opponent sets; None without the Hall of Fame."""
        if not self.hof_size:
            return None
        slots = self.hof_ids.cpu().numpy().copy()
        return slots, np.array([self._hof_eval_slot_gen[s] for s in slots], dtype=np.int64)

    def hof_generations(self):
        """Generations of the filled archive entries, oldest first: the order of :meth:`hof_matrix`."""
        return sorted(self.hof_slot_gen[:self.hof_filled])

    def hof_matrix(self, E=None):
        """Cross-generation matrix of the archive (current individual vs ancestral opponents): fp64
        [filled, filled, 2], entries oldest first (:meth:`hof_generations`).  ``[i, j]`` holds the mean true
        good-team and adversary rewards (rollout columns 0 and 2, the reference's attribution not applied) when the
        good team of entry i plays the adversary of entry j, over E games (default ``envs_per_member``) up to
        ``max_evaluation_steps``.  One structured rollout: the adversaries are the members, the good teams the K
        opponent sets; the initial states come from a Philox stream of their own, so the training run is not
        disturbed.  Replicated: every rank can compute it."""
        if not self.hof_size:
            raise ValueError("hof_matrix needs the Hall of Fame (es_hof_size > 0)")
        E = self.E if E is None else int(E)
        n = self.hof_filled
        order = sorted(range(n), key=lambda s: self.hof_slot_gen[s])
        idx = torch.tensor(order, dtype=torch.int64).to(self.device)
        rows = self.k.gather_rows(self.hof_ring, idx)                        # [n, len(theta_cat)], oldest first
        col = {r: rows[:, o:o + p] for r, (o, p) in self.cols.items()}
        init = self.k.init_states(self.seed, self._hof_matrix_tag, n * n * E, self.device)
        out = self.k.mpe_rollout("adversary_0", col["adversary_0"].contiguous(), col["agent_0"], col["agent_1"],
                                 init.reshape(n, n, E, mpe_spec.INIT_STATE_DIM),
                                 n_cycles=_limit_cycles(self.k, self.args.max_evaluation_steps),
                                 pos_first=self.pos_first, status=self.status)      # [n adversaries, n teams, E, 4]
        self.k.raise_on_status(self.status)
        return out[..., [0, 2]].mean(dim=2).transpose(0, 1).contiguous().to(torch.float64)

    def _sigma_stats(self, role):
        """(mean, min, max, std) of the role's per-parameter sigma after this generation's update over its Linear
        entries (separable NES), None for the isotropic distribution."""
        if not self.separable:
            return None
        st = self.k.weight_stats(self.sigma_rows[role].reshape(1, -1), layout.OBS_DIM[role])
        return tuple(float(x) for x in st[0].cpu().tolist())

    def state_dict(self):
        """Base rows, the update options and search distribution settings, for Adam its moments (its step count is
        the generation count), for separable NES the per-parameter sigmas, for the Hall of Fame its settings, the
        archive ring and its bookkeeping, for guided search its settings, the estimate ring and its bookkeeping
        (the basis is recomputed from them on load), and for novelty search its settings, the characterisation rings
        and their bookkeeping (the probe observations are a function of the seed)."""
        sd = self._base_state()
        sd.update(theta={r: self.theta[r].cpu().clone() for r in ROLES}, es_options=dict(self.options),
                  es_distribution=dict(self.distribution), es_hof=dict(self.hof_opts),
                  es_subspace=dict(self.subspace_opts), es_novelty=dict(self.novelty_opts))
        if self.subspace_k:
            sd.update(subspace_ring=self.subspace_ring.cpu().clone(), subspace_head=self.subspace_head,
                      subspace_filled=self.subspace_filled)
        if self.novelty_w:
            sd.update(novelty_ring=self.novelty_ring.cpu().clone(), novelty_head=self.novelty_head,
                      novelty_filled=self.novelty_filled)
        if self.adam_m is not None:
            sd.update(adam_m=self.adam_m.cpu().clone(), adam_v=self.adam_v.cpu().clone())
        if self.separable:
            sd.update(sigma=self.sigma_cat.cpu().clone())
        if self.lmma_m:
            sd.update(lmma_M=self.lmma_M.cpu().clone(), lmma_p=self.lmma_p.cpu().clone(),
                      lmma_G=self.lmma_G.cpu().clone(), lmma_gen=self.lmma_gen)
        if self.hof_size:
            sd.update(hof_ring=self.hof_ring.cpu().clone(), hof_head=self.hof_head, hof_filled=self.hof_filled,
                      hof_slot_gen=list(self.hof_slot_gen))
        return sd

    def load_state_dict(self, sd):
        """Refuses a checkpoint written with other update options, search distribution, Hall-of-Fame, guided-search or
        novelty-search settings (one without them was written with the defaults)."""
        saved = sd.get("es_options", ES_OPTION_DEFAULTS)
        if saved != self.options:
            raise ValueError(f"checkpoint was written with ES options {saved}, this run uses {self.options}")
        # a checkpoint written before a setting existed was written with its default
        saved = {**ES_DISTRIBUTION_DEFAULTS, **sd.get("es_distribution", {})}
        if saved.get("es_distribution") != "lmma":
            saved.pop("es_lmma_memory", None)
        if saved != self.distribution:
            raise ValueError(f"checkpoint was written with the ES distribution {saved}, this run uses "
                             f"{self.distribution}")
        saved = sd.get("es_hof", ES_HOF_DEFAULTS)
        if saved != self.hof_opts:
            raise ValueError(f"checkpoint was written with the ES Hall of Fame {saved}, this run uses {self.hof_opts}")
        saved = sd.get("es_subspace", ES_SUBSPACE_DEFAULTS)
        if saved != self.subspace_opts:
            raise ValueError(f"checkpoint was written with the ES guided search {saved}, this run uses "
                             f"{self.subspace_opts}")
        saved = sd.get("es_novelty", ES_NOVELTY_DEFAULTS)
        if saved != self.novelty_opts:
            raise ValueError(f"checkpoint was written with the ES novelty search {saved}, this run uses "
                             f"{self.novelty_opts}")
        self._load_base_state(sd)
        for r in ROLES:
            self.theta[r].copy_(sd["theta"][r])
        if self.novelty_w:
            self.novelty_ring.copy_(sd["novelty_ring"])
            self.novelty_head, self.novelty_filled = int(sd["novelty_head"]), int(sd["novelty_filled"])
        if self.separable:
            self.sigma_cat.copy_(sd["sigma"])
        if self.lmma_m:
            self.lmma_M.copy_(sd["lmma_M"])
            self.lmma_p.copy_(sd["lmma_p"])
            self.lmma_G.copy_(sd["lmma_G"])
            self.lmma_gen = int(sd["lmma_gen"])
        if self.hof_size:
            self.hof_ring.copy_(sd["hof_ring"])
            self.hof_head, self.hof_filled = int(sd["hof_head"]), int(sd["hof_filled"])
            self.hof_slot_gen = [int(g) for g in sd["hof_slot_gen"]]
        if self.subspace_k:
            self.subspace_ring.copy_(sd["subspace_ring"])
            self.subspace_head, self.subspace_filled = int(sd["subspace_head"]), int(sd["subspace_filled"])
            if self.subspace_filled:
                self._subspace_basis()
            else:
                self.subspace_U.zero_()
                self.subspace_keff.zero_()
        if self.adam_m is not None:
            self.adam_m.copy_(sd["adam_m"])
            self.adam_v.copy_(sd["adam_v"])


def adapt_sigma(args, hist0, hist1, histadv, gen):
    """Dynamic mutation power (genetic_algorithm.py:323-345 ==
    evolutionary_strategy.py:292-316), including agent_0 growing from
    sigma_agent_1 * 1.2 (Appendix C #6).  Host scalars, mutates ``args``.  The engines run the same
    rule on the device (``cev_generation_end_f64``); this host form serves callers that drive the
    reference's helper functions themselves."""
    def worse(h):
        return gen > 10 and np.mean(h[-10:]) < np.mean(h[-20:-10])
    if worse(hist0):
        args.mutation_power_agent_0 = min(args.mutation_power_agent_1 * 1.2, args.max_mutation_power)
    else:
        args.mutation_power_agent_0 = max(args.mutation_power_agent_0 * 0.95, args.min_mutation_power)
    if worse(hist1):
        args.mutation_power_agent_1 = min(args.mutation_power_agent_1 * 1.2, args.max_mutation_power)
    else:
        args.mutation_power_agent_1 = max(args.mutation_power_agent_1 * 0.95, args.min_mutation_power)
    if worse(histadv):
        args.mutation_power_adversary = min(args.mutation_power_adversary * 1.2, args.max_mutation_power)
    else:
        args.mutation_power_adversary = max(args.mutation_power_adversary * 0.95, args.min_mutation_power)
