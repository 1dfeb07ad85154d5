"""CLI with the reference's flags (``main.py:14-91``) plus build-only options.

    python -m coevonet_b200.main --algorithm=GA --train --game=simple_adversary_v3 ...

``train_GA.sh`` / ``train_ES.sh`` at the repo root pass the reference's
canonical hyper-parameters.  Under ``torchrun`` (one process per GPU) the
population is sharded over the ranks (NCCL).
"""
from __future__ import annotations

import argparse
import os

import torch


def parse_arguments(argv=None):
    p = argparse.ArgumentParser(description="Train a DNN agent using GA or ES (B200-native hot path)")
    p.add_argument("--algorithm", type=str, choices=["GA", "ES"], default="GA")
    p.add_argument("--generations", type=int, default=100)
    p.add_argument("--population", type=int, default=10)
    p.add_argument("--hof_size", type=int, default=20)
    p.add_argument("--game", type=str, choices=["boxing_v2", "pong_v3", "simple_adversary_v3"], default="pong_v3")
    p.add_argument("--initial_mutation_power_agent_0", type=float, default=0.05)
    p.add_argument("--initial_mutation_power_agent_1", type=float, default=0.05)
    p.add_argument("--initial_mutation_power_adversary", type=float, default=0.05)
    p.add_argument("--learning_rate", type=float, default=0.1)
    p.add_argument("--max_timesteps_per_episode", type=int, default=None)
    p.add_argument("--max_evaluation_steps", type=int, default=None)
    p.add_argument("--elites_number", type=int, default=2)
    p.add_argument("--debug", action="store_true")
    p.add_argument("--train", action="store_true")
    p.add_argument("--render", action="store_true")
    p.add_argument("--test", action="store_true")
    p.add_argument("--env_mode", type=str, choices=["AEC"], default="AEC")
    p.add_argument("--precision", type=str, choices=["float32", "float16"], default="float32")
    p.add_argument("--save", action="store_true")
    p.add_argument("--adaptive", action="store_true")
    p.add_argument("--max_mutation_power", type=float, default=0.2)
    p.add_argument("--min_mutation_power", type=float, default=0.001)
    p.add_argument("--fitness_sharing", action="store_true")
    p.add_argument("--ES_model_to_test_agent_0", type=str, default=None)
    p.add_argument("--ES_model_to_test_agent_1", type=str, default=None)
    p.add_argument("--ES_model_to_test_adversary_0", type=str, default=None)
    p.add_argument("--GA_hof_to_test_agent_0", type=str, default=None)
    p.add_argument("--GA_hof_to_test_agent_1", type=str, default=None)
    p.add_argument("--GA_hof_to_test_adversary", type=str, default=None)
    p.add_argument("--play_against_yourself", action="store_true")
    p.add_argument("--average_window", type=int, default=None)
    p.add_argument("--early_stopping", action="store_true")
    p.add_argument("--patience", type=int, default=300)
    p.add_argument("--min_delta", type=float, default=0.1)
    # ---- build-only options (defaults reproduce the reference) -----------------------
    p.add_argument("--envs_per_member", type=int, default=1,
                   help="env instances per (member, opponent) evaluation; the reference plays 1")
    p.add_argument("--no_reference_compat", action="store_true",
                   help="credit each role its own reward, average over all HoF games, seat hof_agent_1 "
                        "correctly (see DESIGN.md, reference quirks)")
    p.add_argument("--init_states", choices=["reference", "device"], default="reference",
                   help="initial env states: the reference's host PCG64 stream, or Philox on the GPU")
    p.add_argument("--device_init", action="store_true",
                   help="draw the GA founders on the device (Philox; same distribution as PyTorch's default "
                        "init) instead of building 3*P nn.Modules on the host; implied for population > 4096")
    p.add_argument("--regenerate_noise", action="store_true",
                   help="ES update: regenerate sigma*z from the Philox key (the reference's exact `noises` array) "
                        "instead of reading it back as members - theta (faster, differs by the rounding of the "
                        "perturbation's add)")
    p.add_argument("--mirrored_sampling", action="store_true",
                   help="ES: members come in antithetic pairs theta +- sigma*z_q sharing one normal draw (Salimans et "
                        "al. 2017); halves the noise generation; needs an even --population")
    p.add_argument("--fitness_shaping", choices=["none", "centered_rank"], default="none",
                   help="ES: weight the update by centered ranks r_i/(P-1) - 0.5 of the global fitness (ties share "
                        "their average rank) instead of the raw fitness.  With --fitness_sharing the ranks are taken "
                        "after its division, which divides every member by the same positive scalar and so does not "
                        "change them")
    p.add_argument("--es_optimizer", choices=["sgd", "adam"], default="sgd",
                   help="ES: step along the update estimate with plain SGD (the reference) or Adam (b1 0.9, b2 0.999, "
                        "eps 1e-8); --learning_rate is then Adam's step size, and 0.1, the reference's SGD default, is "
                        "large for Adam (try 0.01)")
    p.add_argument("--l2_coeff", type=float, default=0.0,
                   help="ES: L2 weight decay, the step follows g = ghat - l2_coeff * theta (with sgd or adam)")
    p.add_argument("--es_distribution", choices=["isotropic", "separable"], default="isotropic",
                   help="ES: search with one mutation power per role (isotropic, the reference) or with one per "
                        "parameter adapted by separable NES (Schaul et al. 2011): sigma starts at "
                        "--initial_mutation_power_*, moves by exp(sigma_learning_rate/2 * g_sigma) every generation and "
                        "stays in [--min_mutation_power, --max_mutation_power]; --learning_rate is then SNES's "
                        "eta_mu (1.0 is the textbook value; the default stays the reference's 0.1).  Not with "
                        "--es_optimizer adam, --l2_coeff or --adaptive")
    p.add_argument("--sigma_learning_rate", type=float, default=None,
                   help="ES, separable: learning rate of log sigma for all roles (default: (3 + ln d) / (5 sqrt d) "
                        "per role, d = its number of Linear parameters)")
    p.add_argument("--es_hof_size", type=int, default=0,
                   help="ES: keep a Hall of Fame of the last H base agents (the founders, then one snapshot per "
                        "generation) and evaluate every member against --es_hof_opponents sets drawn from it; "
                        "0 = off (every member plays the current base agents only, the reference)")
    p.add_argument("--es_hof_opponents", type=int, default=1,
                   help="ES, with --es_hof_size H: opponent sets K per member, 1 <= K <= H.  Set 0 is the current "
                        "base agents, sets 1..K-1 are snapshots drawn uniformly with replacement (the same on every "
                        "rank); each set plays --envs_per_member games, and the reward is the mean over the K x E "
                        "games")
    p.add_argument("--es_subspace_dim", type=int, default=0,
                   help="ES: guided search (Maheswaranathan et al. 2019): put part of the search variance in the "
                        "subspace spanned by the last k update estimates (an orthonormal basis recomputed every "
                        "generation on the device), 0 <= k <= 32; the total variance stays that of the isotropic "
                        "search, so --initial_mutation_power_*, --adaptive and the clamps keep their meaning.  0 = off "
                        "(the isotropic search of the reference).  Not with --es_distribution separable or "
                        "--regenerate_noise")
    p.add_argument("--es_subspace_alpha", type=float, default=None,
                   help="ES, with --es_subspace_dim k: share alpha in (0, 1] of the variance kept isotropic; members "
                        "are theta + sigma (sqrt(alpha) z + sqrt((1 - alpha) d / k_eff) U^T c), d the role's number of "
                        "Linear parameters, k_eff <= k the rank of the basis (default 0.5; 1 = the isotropic search)")
    p.add_argument("--play_discarded_hof_games", action="store_true",
                   help="GA, reference_compat: also simulate the hof_size-1 games per member whose reward the "
                        "reference overwrites (they never reach the fitness; skipped by default)")
    p.add_argument("--seed", type=int, default=1870300, help="run seed of the Philox noise streams")
    p.add_argument("--torch_seed", type=int, default=None, help="torch.manual_seed for the founders")
    p.add_argument("--crossover_rate", type=float, default=0.0,
                   help="GA extension (the reference has no crossover, README.md:47 vs code): probability that a "
                        "child is a uniform crossover of two elites before it is mutated; 0 = reference behaviour")
    p.add_argument("--no_plots", action="store_true")
    p.add_argument("--no_fused_roles", action="store_true",
                   help="play the three roles' evaluation loops as one K1 pass per role on three CUDA streams instead of "
                        "the roles of a generation in one pass (cev_mpe_rollout_roles_f32); same results")
    p.add_argument("--resume", action="store_true",
                   help="continue from <output_dir>/engine_state_rank<r>.pt (written next to the reference-format "
                        ".pth files when --save is set): populations / base rows, HoF ring, sigmas, reward history, "
                        "generation counter, Philox seed, host init-state stream")
    p.add_argument("--log_member_weight_stats", action="store_true",
                   help="ES: per-MEMBER statistics of the perturbed weights every generation (the reference's "
                        "log_weight_statistics, MPE/mpe_agent.py:30-50), reduced on the device")
    return p.parse_args(argv)


class Args:
    """The reference's mutable attribute bag (``main.py:95-142``)."""

    def __init__(self, a):
        self.algorithm = a.algorithm
        self.generations = a.generations
        self.population = a.population
        self.hof_size = a.hof_size
        self.game = a.game
        self.mutation_power_agent_0 = a.initial_mutation_power_agent_0
        self.mutation_power_agent_1 = a.initial_mutation_power_agent_1
        self.mutation_power_adversary = a.initial_mutation_power_adversary
        self.learning_rate = a.learning_rate
        self.max_timesteps_per_episode = a.max_timesteps_per_episode
        self.max_evaluation_steps = a.max_evaluation_steps
        self.elites_number = a.elites_number
        self.adaptive = a.adaptive
        self.max_mutation_power = a.max_mutation_power
        self.min_mutation_power = a.min_mutation_power
        self.fitness_sharing = a.fitness_sharing
        self.early_stopping = a.early_stopping
        self.patience = a.patience
        self.min_delta = a.min_delta
        self.debug = a.debug
        self.train = a.train
        self.test = a.test
        self.render = a.render
        self.env_mode = a.env_mode
        self.precision = a.precision
        self.save = a.save
        self.ES_model_to_test_agent_0 = a.ES_model_to_test_agent_0
        self.ES_model_to_test_agent_1 = a.ES_model_to_test_agent_1
        self.ES_model_to_test_adversary_0 = a.ES_model_to_test_adversary_0
        self.GA_hof_to_test_agent_0 = a.GA_hof_to_test_agent_0
        self.GA_hof_to_test_agent_1 = a.GA_hof_to_test_agent_1
        self.GA_hof_to_test_adversary = a.GA_hof_to_test_adversary
        self.play_against_yourself = a.play_against_yourself
        if a.average_window is not None and a.average_window > a.generations:
            raise ValueError("The average window must be lower than the total number of generations!")
        self.average_window = a.average_window if a.average_window is not None else 50
        self.envs_per_member = a.envs_per_member
        self.reference_compat = not a.no_reference_compat
        self.init_states = a.init_states
        self.device_init = a.device_init or a.population > 4096
        if a.population > 4096 and a.init_states == "reference":
            # the host PCG64 stream costs ~5 us per reset; at this scale draw the states on the device
            self.init_states = "device"
        self.seed = a.seed
        self.play_discarded_hof_games = a.play_discarded_hof_games
        self.update_from_members = not a.regenerate_noise
        self.plots = not a.no_plots
        self.fused_roles = not a.no_fused_roles
        self.resume = a.resume
        self.crossover_rate = a.crossover_rate
        self.log_member_weight_stats = a.log_member_weight_stats
        self.mirrored_sampling = a.mirrored_sampling
        self.fitness_shaping = a.fitness_shaping
        self.es_optimizer = a.es_optimizer
        self.l2_coeff = a.l2_coeff
        self.es_distribution = a.es_distribution
        self.sigma_learning_rate = a.sigma_learning_rate
        self.es_hof_size = a.es_hof_size
        self.es_hof_opponents = a.es_hof_opponents
        self.es_subspace_dim = a.es_subspace_dim
        self.es_subspace_alpha = a.es_subspace_alpha
        from .engine import es_distribution, es_hof, es_options, es_subspace
        es_options(self)                  # ValueError: odd population with mirrored sampling, an ES option with GA
        es_distribution(self)
        es_hof(self)
        es_subspace(self)

    def print_attributes(self, args=None):
        for k, v in vars(self).items():
            print(f"{k.replace('_', ' ').capitalize()}: {v}")


def _init_distributed():
    if "RANK" in os.environ and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        if not dist.is_initialized():
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return True
    return False


def main(argv=None):
    from .evolutionary_strategy import evolution_strategy_train
    from .genetic_algorithm import genetic_algorithm_train
    from .utils.game_logic_functions import initialize_env, play_game
    from .utils.utils_pth_and_plots import create_output_dir, load_agent_for_testing

    ns = parse_arguments(argv)
    args = Args(ns)
    distributed = _init_distributed()
    rank0 = (not distributed) or int(os.environ["RANK"]) == 0
    if rank0:
        print("\nHyperparameters and Parameters:")
        args.print_attributes(args)
        print("\n")
    if ns.torch_seed is not None:
        torch.manual_seed(ns.torch_seed)
    output_dir = create_output_dir(args)

    if args.train:
        if rank0:
            print("Starting Training...")
        env = initialize_env(args)
        if args.algorithm == "GA":
            genetic_algorithm_train(env, env.agents[0], args, output_dir)
        else:
            evolution_strategy_train(env, args, output_dir)
        if rank0:
            print("Training completed.")
        env.close()

    if args.test:
        print("Starting Testing...")
        env = initialize_env(args)
        test_episodes = 10
        agent_0, agent_1, adversary = load_agent_for_testing(args, env)
        tot = [0.0, 0.0, 0.0]
        for _ in range(test_episodes):
            r = play_game(env=env, player1=agent_0.model, player2=agent_1.model, adversary=adversary.model,
                          args=args, eval=True)
            tot = [t + x for t, x in zip(tot, r)]
        print(f"\n Average Reward over {test_episodes}: agent_0 with {tot[0] / test_episodes}, "
              f"agent_1 with {tot[1] / test_episodes}, adversary with {tot[2] / test_episodes}")
        print("Testing completed.")
        env.close()
    if distributed:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
