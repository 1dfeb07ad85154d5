/*
 * coevonet_b200 -- C ABI of the B200-native population-evaluation hot path.
 *
 * The reference (CogSP/CoEvoNet) is pure Python and has no FFI; the drop-in
 * boundary is its Python call surface (SURVEY.md section 8b).  This header is
 * the native boundary underneath that surface: what a binding (ctypes / cffi /
 * pybind) for the hot path binds.  Every entry point cites the reference
 * function whose body it replaces.
 *
 * Conventions
 *  - All pointers are DEVICE pointers owned by the caller unless a parameter is
 *    documented as host memory.  No torch types.  The library allocates nothing
 *    persistent except the per-handle workspace.
 *  - Every compute call is asynchronous on `stream` and returns 0 on success,
 *    <0 on an argument / launch error (text via cev_last_error()).
 *  - Device-detected faults (non-finite activations, the reference's
 *    ValueError at MPE/fcnetwork.py:39-65) are OR-ed into `*status`
 *    (device int32, may be NULL); the caller reads it after synchronising.
 *  - Network rows use the reference's `parameters()` order
 *    (MPE/fcnetwork.py:11-22; SURVEY.md Appendix D) with the row pitch padded
 *    to a multiple of 32 floats: cev_fc_pitch(in_dim).
 *  - Seats are in world / AEC order: 0 = adversary_0, 1 = agent_0, 2 = agent_1.
 */
#ifndef COEVONET_B200_H
#define COEVONET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cev_handle cev_handle;
typedef void* cev_stream;               /* cudaStream_t */

#define CEV_OK 0
#define CEV_ERR_ARG (-1)
#define CEV_ERR_CUDA (-2)
#define CEV_ERR_UNSUPPORTED (-3)

#define CEV_STATUS_NONFINITE 1          /* MPE/fcnetwork.py:39,49,57,65 */

#define CEV_SEAT_ADVERSARY 0
#define CEV_SEAT_AGENT_0 1
#define CEV_SEAT_AGENT_1 2

#define CEV_INIT_STATE_DIM 11           /* goal, adv.xy, a0.xy, a1.xy, lm0.xy, lm1.xy */
#define CEV_ROLLOUT_OUT_DIM 4           /* sum_good, last_good, sum_adv, min_gap */

/* noise kinds (Philox counter word 3 = role | kind << 8) */
#define CEV_KIND_ES 0
#define CEV_KIND_GA 1
#define CEV_KIND_ENV 2
#define CEV_KIND_FRAMES 3
#define CEV_KIND_INIT 4
#define CEV_KIND_XOVER 5
#define CEV_KIND_ES_MIRROR 6            /* ES pair noise under mirrored sampling: member = pair id */
#define CEV_KIND_HOF 7                  /* Co-ES Hall-of-Fame opponent draws: member 0, role 0 */
#define CEV_KIND_ES_SUBSPACE 8          /* Co-ES guided-search coefficients: member = member id, or pair id */

int cev_version(void);
const char* cev_last_error(void);
int cev_create(int device, cev_handle** out);
int cev_destroy(cev_handle* h);
/* number of SMs / co-resident 4-CTA clusters the rollout kernel will use */
int cev_device_info(cev_handle* h, int* n_sm, int* n_clusters);

/* flat-row geometry of FCNetwork(in_dim, 5): 139781 / 138757 and padded pitch */
int cev_fc_dim(int in_dim);
int cev_fc_pitch(int in_dim);
/* DeepQN(c_in, n_actions) row length (Atari/deepqn.py:7-36) and padded pitch */
int cev_dqn_dim(int c_in, int n_actions);
int cev_dqn_pitch(int c_in, int n_actions);

typedef struct {
    int32_t n_cycles;            /* world steps per episode: 25, or floor(limit/3)
                                    under play_MPE's agent-step limit
                                    (utils/game_logic_functions.py:127,195) */
    int32_t integrate_pos_first; /* SURVEY.md Appendix A.4 switch (1 = PettingZoo >= 1.24) */
    int32_t variant;             /* 0 auto (from THIS call's P*K*E), 1 generic kernel, 2 cluster kernel (member
                                    weights resident in shared memory), 3 lockstep kernels (member and opponent
                                    forwards on tcgen05).  A sharded caller passes the variant chosen for the GLOBAL
                                    population (cev_mpe_rollout_plan) so every rank runs the same arithmetic. */
    int32_t reserved;
} cev_rollout_cfg;

/*
 * K1 -- fused MPE rollout, structured form.
 * Replaces the evaluation loops' body: play_game / play_MPE
 * (utils/game_logic_functions.py:123-228) + FCNetwork.forward /
 * determine_action (MPE/fcnetwork.py:37-90) + the simple_adversary_v3 world
 * step, for P members x K opponent sets x E env instances
 * (genetic_algorithm.py:125-217, evolutionary_strategy.py:236-251).
 *
 * Member m sits in `member_seat`; the two other seats (ascending seat order)
 * are filled by opp_a[k], opp_b[k].  init is fp64 [P,K,E,11] (or [K,E,11]
 * shared by all members when init_shared != 0).  out is fp64 [P,K,E,4]:
 * (sum_c r_good, r_good of the last cycle, sum_c r_adv, min top-2 logit gap).
 */
int cev_mpe_rollout_f32(cev_handle* h, int member_seat,
                        const float* members, int P, int64_t member_pitch,
                        const float* opp_a, int64_t opp_a_pitch,
                        const float* opp_b, int64_t opp_b_pitch, int K,
                        const double* init, int init_shared, int E,
                        const cev_rollout_cfg* cfg,
                        double* out, int32_t* status, cev_stream stream);

/*
 * K1 for the roles of one generation in ONE pass (lockstep kernels): the reference evaluates the three
 * roles one after the other (evolutionary_strategy.py:236-251; genetic_algorithm.py:125-217); here their
 * member kernels run back to back on `stream`, their opponent kernels back to back beside them on a
 * share of the SMs, and every role's world step waits only for that role's two kernels.  Results are
 * identical to n_roles calls of cev_mpe_rollout_f32 with variant 3.  Every role has the same P, K, E
 * (n_roles <= 3); a shape below the lockstep threshold is played role by role.
 */
typedef struct {
    int32_t member_seat;         /* 0 adversary_0, 1 agent_0, 2 agent_1 */
    int32_t reserved;
    const float* members;        /* [P, member_pitch] */
    int64_t member_pitch;
    const float* opp_a;          /* [K, opp_a_pitch], the lower of the two other seats */
    int64_t opp_a_pitch;
    const float* opp_b;
    int64_t opp_b_pitch;
    const double* init;          /* fp64 [P,K,E,11] or [K,E,11] (init_shared) */
    double* out;                 /* fp64 [P,K,E,4] */
} cev_rollout_role;

int cev_mpe_rollout_roles_f32(cev_handle* h, int n_roles, const cev_rollout_role* roles,
                              int P, int K, int init_shared, int E,
                              const cev_rollout_cfg* cfg, int32_t* status, cev_stream stream);

/*
 * K1, lockstep kernels (variant 3) with parity instrumentation: the same launches as
 * cev_mpe_rollout_f32, plus -- each optional -- teacher forcing and traces, laid out
 * [n_cycles][3 seats][N = P*K*E episodes]:
 *   forced_actions  int32: actions the world step replays instead of the networks' own
 *                   (the oracle's trace: FCNetwork.forward is then compared logit by logit on
 *                   identical observations, MPE/fcnetwork.py:37-70, SURVEY.md section 7 step 3)
 *   logits_out      fp32 [..][5]: the logits behind every decision (member and opponent forwards
 *                   on tcgen05: 3xTF32 / scaled two-term FP16 with fp32 accumulation)
 *   actions_out     int32: the networks' own first-max decisions (MPE/fcnetwork.py:73-90)
 */
int cev_mpe_rollout_trace_f32(cev_handle* h, int member_seat,
                              const float* members, int P, int64_t member_pitch,
                              const float* opp_a, int64_t opp_a_pitch,
                              const float* opp_b, int64_t opp_b_pitch, int K,
                              const double* init, int init_shared, int E,
                              const cev_rollout_cfg* cfg,
                              const int32_t* forced_actions, float* logits_out, int32_t* actions_out,
                              double* out, int32_t* status, cev_stream stream);

/*
 * Which kernel a structured rollout of this shape uses (variant 0 = the library's choice) and
 * how many kernels one cev_mpe_rollout_f32 call launches.  Host-only, no device work.
 */
int cev_mpe_rollout_plan(cev_handle* h, int P, int K, int E, int n_cycles, int variant,
                         int* variant_used, int* n_launches);

/*
 * Measurement aid: when enabled, the lockstep rollout (variant 3) records CUDA events around every
 * member-forward (which = 0) and opponent-forward (which = 1) kernel launch on the launch stream.
 * cev_kernel_timing_read waits for them, returns the summed device time and the launch count since
 * the last read, and resets the counters.  At most 4096 launches of each kind are kept per read.
 */
int cev_kernel_timing_enable(cev_handle* h, int on);
int cev_kernel_timing_read(cev_handle* h, int which, double* total_ms, int* n_launches);

/*
 * K1 -- indexed form: N independent episodes, episode e played by rows
 * idx[e] = (adversary_0 row, agent_0 row, agent_1 row).  The batched
 * equivalent of N calls of play_game (utils/game_logic_functions.py:215).
 */
int cev_mpe_rollout_indexed_f32(cev_handle* h,
                                const float* w_adv, int64_t adv_pitch,
                                const float* w_a0, int64_t a0_pitch,
                                const float* w_a1, int64_t a1_pitch,
                                const int32_t* idx, const double* init, int N,
                                const cev_rollout_cfg* cfg,
                                double* out, int32_t* status, cev_stream stream);

/*
 * Function-level op: batched FCNetwork.forward + determine_action
 * (MPE/fcnetwork.py:37-90) on caller-supplied observations: sample n uses row
 * idx[n] (row 0 when idx is NULL) and obs[n, 0..in_dim).  logits fp32 [N,5],
 * actions int32 [N] (optional).  Used for logits parity under teacher forcing
 * and by the FCNetwork.forward drop-in.
 */
int cev_fc_forward_f32(cev_handle* h, const float* rows, int64_t pitch, int in_dim,
                       const int32_t* idx, const float* obs, int64_t N,
                       float* logits, int32_t* actions, int32_t* status, cev_stream stream);

/*
 * K3 -- GA re-population.  Replaces mutate_elites (genetic_algorithm.py:32-48)
 * + MPEAgent.clone (MPE/mpe_agent.py:24-28) + Agent.mutate (agent.py:25-29)
 * + "best survives unmutated" (genetic_algorithm.py:255-268).
 * elites: fp32 [E, pitch] gathered elite rows (elite 0 = best).
 * Rows [row0, row0+n_rows) of the NEXT population are written to `out`
 * (local row r = global member row0 + r): global row 0 = elites[0]; global row
 * c >= 1 = elites[(c-1) % E] + sigma * N(0,1), Philox(seed, GA, role, gen,
 * member=c, param).  noise_out (optional) receives the N(0,1) draws.
 *
 * crossover_rate (extension, 0 = the reference: its README.md:47 promises crossover, its code has
 * none, SURVEY.md Appendix C #7): with this probability child c is first recombined -- every
 * parameter from elites[(c-1) % E] or from a second, different elite, one Philox bit per parameter
 * (Philox(seed, XOVER, role, gen, member=c): block 0xFFFFFFFF decides and picks the mate, block j4
 * holds the mask bits of parameters 4*j4 .. 4*j4+3, bit set = first parent) -- and then mutated.
 */
int cev_ga_repopulate_f32(cev_handle* h, const float* elites, int E,
                          int D, int64_t pitch, float sigma, const double* sigma_dev,
                          float crossover_rate,
                          uint64_t seed, int role, uint32_t gen,
                          int64_t row0, int64_t n_rows,
                          float* out, float* noise_out, cev_stream stream);
/*
 * `sigma_dev` (K3, K5, K6; may be NULL): when non-NULL the mutation power is read from this DEVICE
 * fp64 scalar (rounded to fp32 like float(sigma)) instead of the by-value `sigma`: the slot of the
 * generation state cev_generation_end_f64 adapts, so no scalar leaves the device between generations.
 */

/*
 * Elite / Hall-of-Fame extraction (genetic_algorithm.py:240-275): dst[i] = src[idx[i] - row0] when the
 * GLOBAL row id idx[i] (device int64) lies in this rank's block [row0, row0 + n_local), zeros
 * otherwise -- summed over ranks that is the HoF / elite broadcast, with the indices never leaving the
 * device.  n_local < 0: plain gather, dst[i] = src[idx[i] - row0].
 */
int cev_gather_rows_f32(cev_handle* h, const float* src, int64_t pitch,
                        const int64_t* idx, int n, int64_t row0, int64_t n_local,
                        float* dst, cev_stream stream);

/*
 * K4 -- selection.  Replaces np.argsort(fitness)[::-1][:E]
 * (genetic_algorithm.py:223-234): indices of the k largest, descending; any k <= P.
 *   order 0: ties -> lower index, NaN last (= argsort(-f, kind="stable"))
 *   order 1: the reference's expression evaluated with a STABLE ascending sort: ties -> HIGHER
 *            index, NaN first (SURVEY.md Appendix C #18).  NumPy's default kind leaves the order of
 *            ties unspecified (x86-simd-sort on AVX2 / AVX-512 hosts), so this is one admissible
 *            reference outcome, the one of its scalar insertion-sort path.
 */
#define CEV_ORDER_STABLE_DESC 0
#define CEV_ORDER_REFERENCE 1
int cev_select_topk_f64(cev_handle* h, const double* fitness, int64_t P, int k, int order,
                        int64_t* idx_out, cev_stream stream);

/*
 * K5 -- ES perturbation.  Replaces Agent.mutate_ES (agent.py:31-70) for
 * members [row0, row0+n_rows): out[r] = theta + sigma * N(0,1) on Linear
 * parameters only (LayerNorm rows copied), Philox(seed, ES, role, gen, member).
 */
int cev_es_perturb_f32(cev_handle* h, const float* theta, int in_dim,
                       float sigma, const double* sigma_dev, uint64_t seed, int role, uint32_t gen,
                       int64_t row0, int64_t n_rows, int64_t pitch,
                       float* out, float* noise_out, cev_stream stream);

/*
 * K5 for rows whose perturbable parameters are a prefix of the row: DeepQN rows (conv / Linear tensors
 * first, the six BatchNorm vectors last; Atari/deepqn.py:158-172 skips them).  out[r][j] = theta[j] +
 * sigma * N(0,1) for j < d_pert, theta[j] for d_pert <= j < d_total, 0 up to the pitch; same Philox stream
 * as cev_es_perturb_f32.
 */
int cev_es_perturb_prefix_f32(cev_handle* h, const float* theta, int64_t d_pert, int64_t d_total, float sigma,
                              const double* sigma_dev, uint64_t seed, int role, uint32_t gen, int64_t row0,
                              int64_t n_rows, int64_t pitch, float* out, cev_stream stream);

/*
 * K6 -- ES fitness-weighted update.  Replaces compute_weight_update
 * (evolutionary_strategy.py:120-148): delta = lr/(n_total*sigma) *
 * sum_i (sigma*z_i) * fitness_i over members [row0, row0+n_rows), noise
 * regenerated from the Philox key (never read from HBM).  delta is fp32[D]
 * in the full-row layout (zeros on LayerNorm entries); partial sums over a
 * rank's members are all-reduced by the caller.
 */
int cev_es_update_f32(cev_handle* h, const double* fitness, int in_dim,
                      float sigma, const double* sigma_dev, float lr, int64_t n_total,
                      uint64_t seed, int role, uint32_t gen,
                      int64_t row0, int64_t n_rows,
                      float* delta, cev_stream stream);

/*
 * K6, from the materialised members: the same delta with sigma*z_i taken as members[i] - theta (the
 * rows cev_es_perturb_f32 wrote, pitch = cev_fc_pitch(in_dim)), i.e. the `noises` array of
 * compute_weight_update read back at HBM speed instead of regenerated on the ALU.  Differs from
 * cev_es_update_f32 by one rounding of the perturbation's add per term (at most ulp(theta)/2 absolute:
 * about 1e-6 of sigma*z at |theta| ~ 1, sigma = 0.05 -- the same rounding the rollout's members carry).  in_dim = 0 accepts
 * any row layout of `pitch` floats (DeepQN rows): unperturbed entries equal theta and contribute zeros.
 */
int cev_es_update_members_f32(cev_handle* h, const double* fitness, const float* members, int64_t pitch,
                              const float* theta, int in_dim, float sigma, const double* sigma_dev, float lr,
                              int64_t n_total, int64_t n_rows, float* delta, cev_stream stream);

/* theta[j] += delta[j] (evolutionary_strategy.py:259-265) */
int cev_axpy_f32(cev_handle* h, float a, const float* x, float* y, int64_t n, cev_stream stream);

/*
 * Opt-in Co-ES update options (Salimans et al. 2017, "Evolution Strategies as a Scalable Alternative to
 * RL"), extending compute_weight_update (evolutionary_strategy.py:120-148) and Agent.mutate_ES
 * (agent.py:31-70).  None of them is used unless the caller asks for it.
 *
 * K5 with mirrored sampling: members come in pairs; global member c = theta + s*sigma*z_q on the Linear
 * parameters, pair q = c >> 1, s = +1 for even c, -1 for odd c, z_q = Philox(seed, ES_MIRROR, role, gen,
 * member=q).  The odd row is theta + (-(sigma*z)) with the even row's rounded product.  A pair cut by
 * the shard boundary (row0 or row0 + n_rows odd) writes only its local row.  noise_out (optional)
 * receives s*z.  Same arguments as cev_es_perturb_f32.
 */
int cev_es_perturb_mirrored_f32(cev_handle* h, const float* theta, int in_dim,
                                float sigma, const double* sigma_dev, uint64_t seed, int role, uint32_t gen,
                                int64_t row0, int64_t n_rows, int64_t pitch,
                                float* out, float* noise_out, cev_stream stream);

/*
 * K6 with mirrored sampling, noise regenerated: the delta of cev_es_update_f32 for members
 * s_c * sigma*z_{c>>1} (the rows cev_es_perturb_mirrored_f32 writes); z_q is generated once per pair.
 * The terms are accumulated (fmaf) in row order within splits that start on even global rows, so the
 * result is bit-identical to a per-member loop over the same splits.
 */
int cev_es_update_mirrored_f32(cev_handle* h, const double* fitness, int in_dim,
                               float sigma, const double* sigma_dev, float lr, int64_t n_total,
                               uint64_t seed, int role, uint32_t gen,
                               int64_t row0, int64_t n_rows,
                               float* delta, cev_stream stream);

/*
 * Centered-rank fitness shaping of rows [row0, row0 + n_rows) of the GLOBAL fitness[P] (fp64):
 * out[r] = rank_i / (P-1) - 0.5 (0 when P = 1) for i = row0 + r, with the average rank
 * rank_i = #{j : F_j < F_i} + (#{j : F_j == F_i} - 1) / 2 (ties share their average rank, -0.0 == +0.0,
 * every NaN ties with every other NaN and ranks below every number).  Exact in fp64.
 */
int cev_centered_ranks_f64(cev_handle* h, const double* fitness, int64_t P, int64_t row0, int64_t n_rows,
                           double* out, cev_stream stream);

/*
 * Fused ES apply over n_segments (<= 3) FCNetwork rows concatenated in one buffer, segment s of
 * cev_fc_pitch(in_dims[s]) floats (in_dims: HOST array).  delta holds the ascent estimate
 * ghat = 1/(n sigma) sum_i (sigma z_i) F_i (K6 with lr = 1, all-reduced).  g = ghat - l2_coeff * theta, then
 *   CEV_ES_SGD:  theta += lr * g                                        (m, v unused, may be NULL)
 *   CEV_ES_ADAM: m = b1 m + (1-b1) g,  v = b2 v + (1-b2) g g,
 *                theta += alpha_t m / (sqrt(v) + eps),
 *                alpha_t = lr sqrt(1 - b2^t) / (1 - b1^t) in fp64, rounded to fp32; t = updates applied
 *                including this one (>= 1).  (The reference builds an Adam optimizer per agent and never
 *                uses it, MPE/mpe_agent.py:20.)
 * fp32, one IEEE-rounded operation at a time (no FMA contraction; 1-b1 and 1-b2 are rounded fp32
 * differences).  Only the Linear (perturbable) entries change: LayerNorm entries and padding of theta, m
 * and v keep their bits.
 */
#define CEV_ES_SGD 0
#define CEV_ES_ADAM 1
#define CEV_ADAM_BETA1 0.9
#define CEV_ADAM_BETA2 0.999
#define CEV_ADAM_EPS 1e-8
int cev_es_apply_f32(cev_handle* h, float* theta, const float* delta, float* m, float* v, int n_segments,
                     const int* in_dims, int optimizer, double lr, float l2_coeff, int t, cev_stream stream);

/*
 * Separable natural evolution strategies (SNES; Schaul, Glasmachers & Schmidhuber 2011; Wierstra et al.,
 * JMLR 2014): the search distribution of a role is N(mu, diag(sigma^2)), mu = theta, sigma an fp32 row laid
 * out like theta (cev_fc_pitch(in_dim) floats; sigma0 on the Linear entries, 0 on LayerNorm entries and
 * padding).
 *
 * K5: member = theta + fl(sigma[j] * z_j) on the Linear entries (LayerNorm entries copied, padding 0).  z comes
 * from the streams of cev_es_perturb_f32 (mirrored = 0: Philox(ES), member = c) or of
 * cev_es_perturb_mirrored_f32 (mirrored = 1: Philox(ES_MIRROR), member = pair c >> 1, the odd member of a pair
 * takes -z), with their shard and pair-cut rules: with sigma equal to sigma0 on every Linear entry the rows
 * are theirs bit for bit.  noise_out (optional) receives s*z.
 */
int cev_es_perturb_diag_f32(cev_handle* h, const float* theta, const float* sigma, int in_dim, int mirrored,
                            uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                            float* out, float* noise_out, cev_stream stream);

/*
 * K6 of SNES, noise regenerated, over members [row0, row0 + n_rows) of n_total:
 *   g_mu[j]    = fl32(1/n_total) * sum_i F_i z_ij
 *   g_sigma[j] = fl32(1/n_total) * sum_i F_i (z_ij^2 - 1)      (z^2 - 1 = fl(fl(z z) - 1))
 * fp32 fmaf in row order within the splits of cev_es_update_f32 (mirrored = 0) or cev_es_update_mirrored_f32
 * (mirrored = 1: splits start on even global rows), the splits summed in order.  g_mu and g_sigma are
 * fp32[cev_fc_pitch(in_dim)], zeros on LayerNorm entries and padding; partial sums over a rank's members are
 * all-reduced by the caller.  Workspace: 2 * n_split * pitch floats.
 */
int cev_es_update_diag_f32(cev_handle* h, const double* fitness, int in_dim, int mirrored, int64_t n_total,
                           uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, float* g_mu,
                           float* g_sigma, cev_stream stream);

/*
 * SNES apply over n_segments (<= 3) FCNetwork rows concatenated like cev_es_apply_f32 (in_dims and
 * sigma_lr: HOST arrays, sigma_lr[s] = eta_sigma of segment s, fp64, > 0).  On the Linear entries only,
 * one IEEE-rounded fp32 operation at a time, the mu step with the OLD sigma:
 *   theta[j] += fl(lr * fl(sigma[j] * g_mu[j]))
 *   sigma[j]  = clamp(fl(sigma[j] * fl32(exp(0.5 * sigma_lr[s] * g_sigma[j]))), sigma_min, sigma_max)
 * (the exp and its argument in fp64; the clamp is fminf(fmaxf(x, sigma_min), sigma_max)).  LayerNorm entries
 * and padding of theta and sigma keep their bits.
 */
int cev_es_apply_diag_f32(cev_handle* h, float* theta, float* sigma, const float* g_mu, const float* g_sigma,
                          int n_segments, const int* in_dims, float lr, const double* sigma_lr, float sigma_min,
                          float sigma_max, cev_stream stream);

/*
 * Co-ES Hall of Fame: the archive slots of the K opponent sets of generation `gen` (out: DEVICE int64[K]).
 * The archive is a ring whose slots [0, filled) hold snapshots (1 <= filled <= 2^32); `newest` is the slot of
 * the current base agents.  Set 0 is always `newest`; set k >= 1 is drawn uniformly with replacement from the
 * filled slots:
 *   w_k    = word (k - 1) & 3 of Philox(seed; ctr = ((k - 1) >> 2, 0, gen, CEV_KIND_HOF << 8))
 *   out[k] = (uint64(w_k) * filled) >> 32
 * (multiply-shift: slot s is drawn with probability floor or ceil of 2^32 / filled over 2^32, so the bias
 * is at most filled / 2^32).  The key is (seed, gen) alone, so every rank draws the same slots.
 */
int cev_es_hof_opponents_i64(cev_handle* h, uint64_t seed, uint32_t gen, int K, int64_t filled, int64_t newest,
                             int64_t* out, cev_stream stream);

/*
 * Co-ES guided search in the subspace of the last k update estimates (Guided ES, Maheswaranathan et al. 2019;
 * the subspace built from the ES's own past updates as in ASEBO, Choromanski et al. 2019).  U is an orthonormal
 * basis fp32 [k][ldu] of k_eff <= k directions laid out like theta (zero on LayerNorm entries and padding).
 *
 * K5: on the Linear entries, with d = the number of Linear entries of the row (cev_fc_dim(in_dim) minus the
 * LayerNorm entries), A = fp32(sqrt(alpha)) and B = fp32(sqrt((1 - alpha) * d / k_eff)) (fp64, then rounded):
 *   s_j   = sum_{m < k_eff} fl(U[m][j] * c_m)      (fp32, one rounding per operation, m = 0, 1, ... in order,
 *                                                   starting from +0)
 *   eps_j = fl(fl(A * z_j) + fl(B * s_j)),   member = theta + fl(sigma * eps_j)
 * and the odd member of a mirrored pair is theta + (-fl(sigma * eps_j)).  LayerNorm entries are copied, padding is 0.
 * z is the stream of cev_es_perturb_f32 (mirrored = 0) or cev_es_perturb_mirrored_f32 (mirrored = 1), with their
 * shard and pair-cut rules.  c holds k normals per unit u (the member id, or the pair id c >> 1 when mirrored):
 *   c_{4 m4 + t} = normal t of the Box-Muller pairs of Philox(seed; ctr = (m4, u, gen, role | CEV_KIND_ES_SUBSPACE << 8)),
 * the transform of the K5 stream, so c does not depend on k_eff (member i uses the first k_eff of its normals).
 * E||eps||^2 = d, the total variance of the isotropic search.  k_eff is read from the DEVICE int k_eff[0]
 * (clamped to [0, k]); when k_eff = 0 or alpha = 1 (B = 0) eps = z and the rows are those of the isotropic K5 bit
 * for bit.  noise_out (optional, [n_rows][pitch]) receives s*z and coef_out (optional, [n_rows][k]) s*c, s = -1 for
 * the odd member of a mirrored pair and +1 otherwise.  1 <= k <= CEV_SUBSPACE_MAX_DIM, 0 < alpha <= 1,
 * ldu >= pitch a multiple of 4.
 */
#define CEV_SUBSPACE_MAX_DIM 32
int cev_es_perturb_subspace_f32(cev_handle* h, const float* theta, int in_dim, float sigma, const double* sigma_dev,
                                const float* U, int64_t ldu, int k, const int* k_eff, double alpha, int mirrored,
                                uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                                float* out, float* noise_out, float* coef_out, cev_stream stream);

/*
 * The orthonormal basis of the guided-search subspace, for n_segments (<= 3) FCNetwork rows concatenated like
 * cev_es_apply_f32 (in_dims: HOST array; n = the summed pitches).  ring: DEVICE fp32 [k][n], slots [0, filled)
 * filled, slot `newest` the newest estimate.  Per segment, over its Linear entries, with the columns
 * D_a = ring[(newest - a) mod k] for a < filled (newest first):
 *   CholeskyQR2 in fp64: G = D^T D (fp64 products of the fp32 values, summed per column chunk in column order, the
 *   chunks in order); a right-looking Cholesky of G over a = 0, 1, ... that DROPS column a when its squared
 *   residual is <= 1e-8 of G[a][a] (its residual norm is <= 1e-4 of its own norm; a zero or non-finite column is
 *   always dropped); U = fp32(D R^-1) on the kept columns, in their order; then the same once more on U.
 * U (out): DEVICE fp32 [k][n], rows [0, k_eff) orthonormal, the other rows and every LayerNorm / padding entry 0;
 * a dropped estimate never enters U, even when it holds an inf or a NaN.
 * k_eff (out): DEVICE int32 [n_segments].  Deterministic; workspace (n_segments * (ceil(max pitch / 4096) + 1) * k^2
 * doubles).  ring and U must not overlap.
 */
int cev_es_subspace_basis_f32(cev_handle* h, const float* ring, int k, int newest, int filled, int n_segments,
                              const int* in_dims, float* U, int* k_eff, cev_stream stream);

/*
 * Co-ES limited-memory matrix adaptation (LM-MA-ES, Loshchilov, Glasmachers & Beyer, IEEE TEC 23(2), 2019).  Per
 * role m direction vectors M fp32 [m][ldm] laid out like theta (zero on LayerNorm entries and padding), their Gram
 * G fp64 [m][ldg], an evolution path p and sigma in CEV_GS_SIGMA + role.  z_i is member i's normals of the stream of
 * cev_es_perturb_f32 on the Linear entries; at generation g the first k = min(g, m) vectors are in use.
 *
 * Projection and coefficients: s_l = m_l . z_i for l < k, with fp32 x fp32 products accumulated in fp64 one add at a
 * time, in column order within fixed chunks of 2048 columns from +0, and the chunks summed in order, so s does not
 * depend on row0, n_rows or the grid.  Then, every operation one fp64 rounding (cd: HOST fp64 [k], c_d,j):
 *   alpha = 1, beta = 0; for j < k: q = alpha s_j + sum_{l<j} beta_l G[j][l] (l in order);
 *   beta_l *= (1 - cd[j]) for l < j; beta_j = cd[j] q; alpha *= (1 - cd[j])
 * beta (out): DEVICE fp32 [n_rows][k]; part: DEVICE workspace fp64 [ceil(fc_dim / 2048)][n_rows][k]; s_out
 * (optional): fp64 [n_rows][k].  A non-finite s or beta sets CEV_STATUS_NONFINITE in *status (optional).
 */
int cev_es_lmma_project_f32(cev_handle* h, const float* M, int64_t ldm, int k, const double* G, int ldg,
                            const double* cd, int in_dim, uint64_t seed, int role, uint32_t gen, int64_t row0,
                            int64_t n_rows, double* part, float* beta, double* s_out, int* status, cev_stream stream);

/*
 * LM-MA K5: on the Linear entries eps_j = fl(fl(alpha * z_j) + S_j), S_j = sum_{l < k} fl(M[l][j] * beta[i][l])
 * (fp32, l in order, from +0), member = theta + fl(fp32(sigma_dev[0]) * eps_j); LayerNorm entries copied, padding 0.
 * This is cev_es_perturb_subspace_f32's arithmetic with A = alpha and B = 1.  beta: DEVICE fp32 [n_rows][k] (row r =
 * member row0 + r).  1 <= k <= CEV_SUBSPACE_MAX_DIM, ldm >= pitch a multiple of 4.
 */
int cev_es_perturb_lmma_f32(cev_handle* h, const float* theta, int in_dim, const double* sigma_dev, const float* M,
                            int64_t ldm, int k, const float* beta, float alpha, uint64_t seed, int role, uint32_t gen,
                            int64_t row0, int64_t n_rows, int64_t pitch, float* out, cev_stream stream);

/*
 * LM-MA weighted recombination over this rank's rows [row0, row0 + n_rows): ids DEVICE int64 [mu] (the selected
 * members, best first) and w DEVICE fp32 [mu] (the weight of each rank).  zbar (out, fp32 [pitch]) = sum over the ranks
 * a whose member is local, in rank order within 8 fixed splits of [0, mu), of fma(w_a, z_id[j], .) in fp64 (exact
 * products), the splits summed in order, rounded to fp32 once (0 off the Linear entries); betabar (out, fp32 [k]) =
 * fp32(sum in rank order of fma(w_a, beta[id - row0][l], .)) in fp64.  Members of other ranks add nothing, so the sum
 * over ranks of zbar / betabar is the population's.  part: DEVICE workspace fp64 [8][pitch].
 */
int cev_es_lmma_reduce_f32(cev_handle* h, const int64_t* ids, const float* w, int mu, const float* beta, int k,
                           int in_dim, uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows,
                           double* part, float* zbar, float* betabar, cev_stream stream);

/*
 * LM-MA apply over n_segments (<= 3) FCNetwork rows concatenated like cev_es_apply_f32 (in_dims, alpha, c_sigma,
 * mu_w: HOST arrays [n_segments]; c_c: HOST fp64 [n_segments][m]).  M: DEVICE fp32 [m][n], p, theta, zbar: fp32 [n],
 * betabar: fp32 [n_segments][m] (the first k of each used).  On the Linear entries, every operation one fp64 rounding
 * and every store one fp32 rounding:
 *   dbar = alpha zbar + sum_{l<k} betabar_l M[l] (M before its update); theta += (c_m fp32(sigma)) dbar;
 *   p = (1 - c_s) p + sqrt(mu_w c_s (2 - c_s)) zbar;  M[l] = (1 - c_c,l) M[l] + sqrt(mu_w c_c,l (2 - c_c,l)) zbar, l < m
 * then G (out, DEVICE fp64 [n_segments][m][m]) = the Gram of the new M and |p|^2 (fp64 products of the fp32 values,
 * column order within chunks of 4096 columns, the chunks in order), and
 *   sigma = clamp(sigma exp(c_s / 2 (|p|^2 / n - 1)), sigma_min, sigma_max)   (n: the row's Linear entries)
 * into gstate[CEV_GS_SIGMA + s]; stats (out, DEVICE fp64 [n_segments][2]) = (|p|^2 / n, sigma).  A non-finite |p|^2 or
 * Gram entry sets CEV_STATUS_NONFINITE and leaves sigma.  part: DEVICE workspace fp64
 * [n_segments][ceil(max pitch / 4096)][m (m + 1) / 2 + 1].
 */
int cev_es_lmma_apply_f32(cev_handle* h, float* theta, float* M, int m, int k, float* p, const float* zbar,
                          const float* betabar, int n_segments, const int* in_dims, const double* alpha,
                          const double* c_sigma, const double* mu_w, double c_m, const double* c_c, double* G,
                          double* gstate, double sigma_min, double sigma_max, double* part, double* stats,
                          int* status, cev_stream stream);

/*
 * Co-ES novelty search (NS-ES / NSR-ES, Conti et al. 2018) on a policy-space behaviour characterisation (the
 * "behavioural embedding" of Parker-Holder et al. 2020): a member is characterised by its action distributions on
 * CEV_NOVELTY_PROBES fixed probe observations, so the characterisation does not depend on the opponents it played.
 *
 * Probe observations: obs fp32 [n][in_dim(seat)] = what seat `seat` (0 adversary_0, 1 agent_0, 2 agent_1) observes
 * in the world state of init record i (fp64 [n][CEV_INIT_STATE_DIM], zero velocities): the rollout's observation,
 * fp64 differences rounded to fp32.
 */
#define CEV_NOVELTY_PROBES 32
#define CEV_NOVELTY_BC_DIM 160          /* CEV_NOVELTY_PROBES * 5 actions */
#define CEV_NOVELTY_MAX_K 32
#define CEV_NOVELTY_MAX_ARCHIVE 32768
int cev_novelty_probe_obs_f32(cev_handle* h, const double* init, int64_t n, int seat, float* obs, cev_stream stream);

/*
 * Behaviour characterisation of P FCNetwork rows (pitch: any multiple of 4 floats >= cev_fc_dim(in_dim); the floats
 * past the network are never read) on the probe observations probe_obs fp32 [CEV_NOVELTY_PROBES][in_dim]:
 *   bc[m][5 p + a] = softmax(logits of row m on probe p)[a] = exp(l_a - max l) / sum_b exp(l_b - max l)
 * fp32 (FFMA forward; the logits within a few ulps of a float32 forward, not bit for bit), row m of bc at
 * m * bc_pitch (bc_pitch >= CEV_NOVELTY_BC_DIM, so a row can be a slot of an archive ring).  A non-finite logit
 * sets CEV_STATUS_NONFINITE in *status (optional).  Each row is read from global memory once; deterministic, and a
 * row's result does not depend on P or on the other rows.
 */
int cev_novelty_bc_f32(cev_handle* h, const float* rows, int64_t pitch, int in_dim, int64_t P, const float* probe_obs,
                       float* bc, int64_t bc_pitch, int32_t* status, cev_stream stream);

/*
 * k-NN novelty of n characterisations bc fp32 [n][CEV_NOVELTY_BC_DIM] against the archive ring fp32
 * [>= filled][CEV_NOVELTY_BC_DIM], slots [0, filled) filled (1 <= filled <= CEV_NOVELTY_MAX_ARCHIVE,
 * 1 <= k <= CEV_NOVELTY_MAX_K):
 *   dist_e = sqrt(sum_t (x_t - y_et)^2)   fp64, t = 0 .. 159 in order, one rounding per operation (no FMA)
 *   novelty[i] = (sum of the k_eff smallest dist_e, in ascending order of (dist_e, e)) / k_eff,
 *                k_eff = min(k, filled), summed from +0 one rounded add at a time
 * novelty: DEVICE fp64 [n].  Exact given finite inputs (the value does not depend on how ties are broken).  A NaN
 * distance (a NaN in bc or in the ring) is never among the k smallest; with fewer than k_eff other entries the sum
 * takes +inf for the missing ones, so such a member's novelty is +inf, where the restatement of the formula gives
 * NaN.  cev_novelty_bc_f32 has set the status word for a NaN characterisation by then.
 */
int cev_novelty_knn_f64(cev_handle* h, const float* bc, int64_t n, const float* ring, int64_t filled, int k,
                        double* novelty, cev_stream stream);

/*
 * Co-GA novelty search (Lehman & Stanley 2011, with a GA on deep networks as in Such et al. 2017): the novelty of
 * a member is measured against the whole current population plus an archive of earlier members' characterisations.
 *
 * k-NN novelty of the n members x fp32 [n][x_pitch] (characterisations of the global rows row0 .. row0 + n - 1)
 * against the candidates: the P population rows pop fp32 [P][pop_pitch] (candidate index c in [0, P); e.g. one
 * role's column of a gathered [P][3][160] block, pop_pitch = 480) and the archive slots ring fp32 [filled][160]
 * (index P + s).  A member is never its own candidate (excluded by id, not by value).  Per (member, candidate):
 *   e_t = fl(q_t - x_t), s = fmaf(e_t, e_t, s)   fp32 from +0, t = 0 .. 159 in order;  dist = sqrt(s) fp32 (rounded)
 * The candidates are ordered by (dist, index), a NaN dist after every number; with k_eff = min(k, P - 1 + filled)
 *   novelty[i] = (sum of the k_eff smallest dist, in that order, fp64 from +0, one rounding per add) / k_eff
 * (a NaN among them makes the novelty NaN).  1 <= k <= CEV_NOVELTY_MAX_K, 0 <= filled <= CEV_NOVELTY_MAX_ARCHIVE,
 * P - 1 + filled >= 1, row0 + n <= P; pitches are multiples of 4 floats >= 160 and the rows 16-byte aligned.
 * `splits` candidate ranges are searched by separate CTAs (0 = chosen from the shape, clamped to the candidate
 * tiles) and merged; the result does not depend on it, on the tiling or on row0's block, so a sharded population
 * gives the values of an unsharded one.  Deterministic.  novelty: DEVICE fp64 [n].  Uses the handle's workspace.
 */
#define CEV_KIND_GA_NOVELTY 9           /* Co-GA novelty archive draws: member 0, role = the role */
int cev_ga_novelty_knn_f64(cev_handle* h, const float* x, int64_t x_pitch, int64_t n, int64_t row0, const float* pop,
                           int64_t pop_pitch, int64_t P, const float* ring, int64_t filled, int k, int splits,
                           double* novelty, cev_stream stream);

/*
 * The m population ids whose characterisations enter the archive of `role` after generation gen's selection, in
 * draw order: id_j = (uint64(w_j) * P) >> 32 with w_j word (j & 3) of the Philox block (j >> 2, 0, gen,
 * role | CEV_KIND_GA_NOVELTY << 8) keyed by seed.  out: DEVICE int64 [m].  1 <= P <= 2^32.
 */
int cev_ga_novelty_draw_i64(cev_handle* h, uint64_t seed, uint32_t gen, int role, int m, int64_t P, int64_t* out,
                            cev_stream stream);

/*
 * Co-GA safe mutations through output gradients (SM-G-SUM, Lehman, Chen, Clune & Stanley, GECCO 2018): each
 * parameter's mutation is divided by how strongly the network's logits respond to it on the probe observations.
 *
 * Scale rows of E parent rows fp32 [E][pitch] of in_dim 8 or 10 (e.g. the gathered elites) on the 32 probe
 * observations probe_obs fp32 [32][in_dim] (cev_novelty_probe_obs_f32).  With y_k(x_t), k = 0..4, the logits of
 * the FCNetwork on probe t (ReLU' = [input > 0]; LayerNorm biased-variance, eps 1e-5), for every entry j < D =
 * cev_fc_dim(in_dim), LayerNorm gains and biases included:
 *   G_kj = sum_t dy_k(x_t) / dW_j,  s_j = sqrt(sum_k G_kj^2),
 *   c_j  = 1 if s_j == 0 (no logit responds to the entry), else fl32(1 / max(s_j, floor))
 * written to scale fp32 [E][scale_pitch]; entries [D, scale_pitch) are 0.  FP32 with every sum in a fixed order:
 * deterministic, and row e does not depend on E.  A non-finite logit or gradient sets CEV_STATUS_NONFINITE in
 * *status (may be NULL).  floor: finite and > 0.  Pitches are multiples of 4 floats >= D, rows 16-byte aligned.
 * Five kernel launches; uses the handle's workspace (about 640 KB per parent).
 */
int cev_ga_safe_scale_f32(cev_handle* h, const float* rows, int64_t pitch, int in_dim, int E, const float* probe_obs,
                          float floor, float* scale, int64_t scale_pitch, int32_t* status, cev_stream stream);

/*
 * K3 with safe mutations: cev_ga_repopulate_f32 (same arguments, same Philox streams and crossover) where the
 * mutation of parameter j of child c >= 1 is fl(p_j + fl(fl(sigma * z_j) * c_j)), c_j from scale fp32 [E][pitch]
 * (cev_ga_safe_scale_f32 of the same elites) of the elite p_j was copied from.  A scale row of ones gives
 * cev_ga_repopulate_f32's rows bit for bit.
 */
int cev_ga_repopulate_safe_f32(cev_handle* h, const float* elites, const float* scale, int E, int D, int64_t pitch,
                               float sigma, const double* sigma_dev, float crossover_rate, uint64_t seed, int role,
                               uint32_t gen, int64_t row0, int64_t n_rows, float* out, float* noise_out,
                               cev_stream stream);

/*
 * K7 -- fitness-sharing distances.  Replaces the distance loop of
 * diversity_penalty (utils/game_logic_functions.py:12-37):
 * d[i] = || pop[i] - ref ||_2 over the perturbable (Linear) parameters.
 */
int cev_diversity_dist_f32(cev_handle* h, const float* pop, int64_t n_rows,
                           int64_t pitch, const float* ref, int in_dim,
                           float* dist, cev_stream stream);

/*
 * Per-member statistics of the perturbable weights.  Replaces MPEAgent.log_weight_statistics
 * (MPE/mpe_agent.py:30-50; called once per perturbed member from Agent.mutate_ES, agent.py:66):
 * out fp32 [n_rows, 4] = (mean, min, max, population std) of get_perturbable_weights().
 */
int cev_weight_stats_f32(cev_handle* h, const float* rows, int64_t n_rows, int64_t pitch, int in_dim,
                         float* out, cev_stream stream);

/*
 * End of a generation, on the device (SURVEY.md 8f N1).  Replaces the tail of the training loops:
 * the mean of the evaluation games (evaluate_current_weights, genetic_algorithm.py:12-29,
 * evolutionary_strategy.py:22-59), rewards_over_generations.append, the adaptive mutation power
 * (genetic_algorithm.py:323-345, evolutionary_strategy.py:292-316; NumPy's mean order, agent_0
 * growing from sigma_agent_1 * 1.2) and the early-stopping counters
 * (evolutionary_strategy.py:318-354).
 *
 * eval_out: fp64 [n_games, 4], the rollout output of the evaluation games.  gstate: DEVICE fp64
 * array of cev_generation_state_doubles(hist_capacity) entries, roles in the order agent_0, agent_1,
 * adversary_0:
 */
#define CEV_GS_GEN 0          /* generations finished so far                                   */
#define CEV_GS_SIGMA 1        /* [3] current mutation power (the sigma_dev slots of K3/K5/K6)  */
#define CEV_GS_BEST 4         /* [3] best evaluation reward (early stopping), init -inf        */
#define CEV_GS_STALE 7        /* [3] generations without improvement                           */
#define CEV_GS_STOP 10        /* 0, or 1 + role index of the role that triggered early stopping */
#define CEV_GS_STOP_GEN 11
#define CEV_GS_LAST_EVAL 12   /* [3] evaluation rewards of the generation just finished         */
#define CEV_GS_HIST 16        /* [hist_capacity][3] evaluation rewards, then [hist_capacity+1][3]
                                 mutation-power history (entry 0 = the initial sigma)          */
int cev_generation_state_doubles(int hist_capacity);
int cev_generation_end_f64(cev_handle* h, const double* eval_out, int n_games, int agent_step_limit,
                           int reference_compat, double* gstate, int hist_capacity, int adaptive,
                           double sigma_max, double sigma_min, int early_stopping, double min_delta,
                           int patience, cev_stream stream);

/*
 * K2 -- grouped per-member DeepQN forward.  Replaces DeepQN.forward
 * (Atari/deepqn.py:39-48): frames u8 [P,B,C,84,84]; logits fp32 [P,B,A];
 * actions int32 [P,B] (first maximum, Atari/deepqn.py:55-60).
 */
int cev_deepqn_forward(cev_handle* h, const float* members, int P, int64_t pitch,
                       const uint8_t* frames, int B, int c_in, int n_actions,
                       float* logits, int32_t* actions, cev_stream stream);

/*
 * N4 -- synthetic Atari-like emulator around K2 (SURVEY.md 8f).  The reference's Atari rollout
 * (utils/game_logic_functions.py:48-53,84-119) is dead code and needs ROMs; these two entry points give
 * its wrapper chain a deterministic stand-in: cev_atari_synth_step_u8 writes frame `t` of episodes
 * ep0 .. ep0+n-1 into slot t % 4 of a u8 ring [n, 4, 84*84] (Philox bytes keyed by episode, cycle and
 * the joint action a_first + 32 a_second; t = 0 needs no actions) and the zero-sum reward
 * r_first in [-1, 1) of that emulator step; cev_atari_observe_u8 builds what the agent `seat`
 * (0 first_0, 1 second_0) observes after t steps: u8 [n, 6, 84*84] = frame_stack_v1(4) (oldest first,
 * zeros before the first frames) + agent_indicator_v0 planes (255 on the agent's own plane).
 */
int cev_atari_synth_step_u8(cev_handle* h, uint64_t seed, int64_t ep0, int64_t n, int t,
                            const int32_t* a_first, const int32_t* a_second, uint8_t* ring,
                            float* r_first, cev_stream stream);
int cev_atari_observe_u8(cev_handle* h, const uint8_t* ring, int64_t n, int t, int seat,
                         uint8_t* obs, cev_stream stream);

/*
 * Founder initialisation on the device.  Replaces create_agent -> MPEAgent -> FCNetwork
 * default init (utils/game_logic_functions.py:58-64, MPE/fcnetwork.py:11-22) for rows
 * [row0, row0+n_rows): Linear weight/bias ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)), LayerNorm
 * gamma = 1, beta = 0, Philox(seed, INIT, role, member, param).
 */
int cev_fc_init_f32(cev_handle* h, int in_dim, uint64_t seed, int role, int64_t row0, int64_t n_rows,
                    int64_t pitch, float* out, cev_stream stream);

/* device-side synthetic inputs (bench / tests): initial env states drawn
 * U(-1,1)^2 + goal in {0,1} (Appendix A.3 distribution, Philox stream; records
 * rec0 .. rec0+n-1 of stream `stream_id`, so shards generate their own slice)
 * and uint8 frames. */
int cev_init_states_f64(cev_handle* h, uint64_t seed, uint32_t stream_id,
                        int64_t rec0, int64_t n, double* out, cev_stream stream);
int cev_random_frames_u8(cev_handle* h, uint64_t seed, int64_t n_bytes,
                         uint8_t* out, cev_stream stream);
/* raw Philox words for bit-exact RNG checks: out u32 [n_members, n4, 4] */
int cev_philox_words(cev_handle* h, uint64_t seed, int kind, int role, uint32_t gen,
                     int64_t member0, int64_t n_members, int64_t n4,
                     uint32_t* out, cev_stream stream);

/* FP32 FMA-pipe peak micro-benchmark (SURVEY.md section 8d: the FP32 roofline
 * denominator is measured, not assumed).  Returns achieved TFLOP/s in *tflops
 * (host pointer); mode 0 = scalar FFMA, 1 = packed FFMA2. */
int cev_fp32_peak(cev_handle* h, int mode, double* tflops, cev_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* COEVONET_B200_H */
