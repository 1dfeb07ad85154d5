// K3-K7: population-level GA / ES kernels over flat parameter rows.
// All are streaming kernels (HBM-bound or Philox-ALU-bound): 128-bit accesses,
// one float4 of parameters per thread, grids sized from the data.
#include "common.cuh"
#include "es_perturb.cuh"

namespace cev {

constexpr int PT = 256;

// ---------------------------------------------------------------------------
// K3  GA re-population   (genetic_algorithm.py:32-48,255-290; agent.py:25-29)
// child c>=1 = elites[(c-1)%E] + sigma*z ; child 0 = elites[0] unmutated.
// Every parameter is mutated (LayerNorm gamma/beta too, Appendix C #8).
// mul and add are rounded separately, like `param.data += noise`.
// ---------------------------------------------------------------------------
// Optional uniform crossover (BASELINE north star item 3; the reference's README.md:47 promises crossover, its
// code has none -- SURVEY.md Appendix C #7 -- so this is an extension, off by default): with probability
// `xrate` child c takes every parameter from parent A = elites[(c-1) % E] or from a second, different elite B
// (one Philox bit per parameter), then mutates as usual.  Philox kind CEV_KIND_XOVER: block (0xFFFFFFFF, c, gen)
// decides (word 0 < xrate * 2^32) and picks the mate (word 1), block (j4, c, gen) holds the four mask bits.
__global__ void __launch_bounds__(PT) ga_repopulate_kernel(
    const float* __restrict__ elites, int E, int D, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0,
    float xrate, uint32_t xtag,
    float* __restrict__ out, float* __restrict__ noise_out) {
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const int64_t r = blockIdx.x;
    const int64_t c = row0 + r;                       // global member id
    const int j4 = blockIdx.y * PT + threadIdx.x;
    __shared__ int64_t mate_s;
    int64_t mate = -1;
    if (xrate > 0.f && E >= 2) {                       // uniform per CTA: one child per blockIdx.x
        if (threadIdx.x == 0) {
            int64_t m = -1;
            if (c != 0) {
                const U4 y = philox4x32_10(U4{0xFFFFFFFFu, (uint32_t)c, gen, xtag}, keys);
                if ((double)y.x < (double)xrate * 4294967296.0)
                    m = ((c - 1) % E + 1 + (int64_t)(y.y % (uint32_t)(E - 1))) % E;
            }
            mate_s = m;
        }
        __syncthreads();
        mate = mate_s;
    }
    if ((int64_t)j4 * 4 >= pitch) return;
    const int64_t parent = (c == 0) ? 0 : (c - 1) % E;
    const float4 pv = *reinterpret_cast<const float4*>(elites + parent * pitch + (int64_t)j4 * 4);
    float p[4] = {pv.x, pv.y, pv.z, pv.w};
    if (mate >= 0) {
        const float4 qv = *reinterpret_cast<const float4*>(elites + mate * pitch + (int64_t)j4 * 4);
        const U4 x = philox4x32_10(U4{(uint32_t)j4, (uint32_t)c, gen, xtag}, keys);
        if (!(x.x & 1u)) p[0] = qv.x;
        if (!(x.y & 1u)) p[1] = qv.y;
        if (!(x.z & 1u)) p[2] = qv.z;
        if (!(x.w & 1u)) p[3] = qv.w;
    }
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (c != 0) {
        normal4(keys, tag, gen, (uint32_t)c, (uint32_t)j4, z);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int j = j4 * 4 + i;
            if (j < D) p[i] = __fadd_rn(p[i], __fmul_rn(sigma, z[i]));
            else { p[i] = 0.f; z[i] = 0.f; }
        }
    }
    *reinterpret_cast<float4*>(out + r * pitch + (int64_t)j4 * 4) = make_float4(p[0], p[1], p[2], p[3]);
    if (noise_out)
        *reinterpret_cast<float4*>(noise_out + r * pitch + (int64_t)j4 * 4) = make_float4(z[0], z[1], z[2], z[3]);
}

// ---------------------------------------------------------------------------
// K5  ES perturbation   (agent.py:31-70): Linear parameters only.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(K5T, 10) es_perturb_kernel(
    const float* __restrict__ theta, int in_dim, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0,
    float* __restrict__ out, float* __restrict__ noise_out) {
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r = blockIdx.x;
    const int64_t c = row0 + r;
    const int j4 = blockIdx.y * K5T + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    es_perturb_float4<false>(theta, o, j4, ScalarSigma{sigma}, keys, tag, gen, (uint32_t)c, out + r * pitch, nullptr,
                             noise_out ? noise_out + r * pitch : nullptr, nullptr);
}

// K5 under mirrored sampling (Salimans et al. 2017): one CTA row per PAIR q of the local block, members 2q and
// 2q+1 from one normal draw (half the Philox / Box-Muller work of es_perturb_kernel).  Local row r holds global
// member row0 + r; the first / last pair writes only its local row when row0 / row0 + n_rows is odd.
__global__ void __launch_bounds__(K5T, 10) es_perturb_mirrored_kernel(
    const float* __restrict__ theta, int in_dim, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows,
    float* __restrict__ out, float* __restrict__ noise_out) {
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t q = (row0 >> 1) + blockIdx.x;
    const int64_t r_plus = 2 * q - row0, r_minus = r_plus + 1;        // local rows of members 2q, 2q+1
    const bool has_plus = r_plus >= 0, has_minus = r_minus < n_rows;
    const int j4 = blockIdx.y * K5T + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    es_perturb_float4<true>(theta, o, j4, ScalarSigma{sigma}, keys, tag, gen, (uint32_t)q,
                            has_plus ? out + r_plus * pitch : nullptr, has_minus ? out + r_minus * pitch : nullptr,
                            noise_out && has_plus ? noise_out + r_plus * pitch : nullptr,
                            noise_out && has_minus ? noise_out + r_minus * pitch : nullptr);
}

// K5 of separable NES: member = theta + fl(sigma[j] z_j) with the per-parameter sigma row, on the CTA grid and
// Philox streams of es_perturb_kernel (MIRROR = false) / es_perturb_mirrored_kernel (MIRROR = true), so a row of
// sigma0 gives their members bit for bit.
template <bool MIRROR>
__global__ void __launch_bounds__(K5T, 10) es_perturb_diag_kernel(
    const float* __restrict__ theta, const float* __restrict__ sigma, int in_dim, int64_t pitch,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows,
    float* __restrict__ out, float* __restrict__ noise_out) {
    const FcOffsets o = fc_offsets(in_dim);
    const int j4 = blockIdx.y * K5T + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    const RowSigma sig{sigma};
    if (!MIRROR) {
        const int64_t r = blockIdx.x;
        es_perturb_float4<false>(theta, o, j4, sig, keys, tag, gen, (uint32_t)(row0 + r), out + r * pitch, nullptr,
                                 noise_out ? noise_out + r * pitch : nullptr, nullptr);
    } else {
        const int64_t q = (row0 >> 1) + blockIdx.x;
        const int64_t r_plus = 2 * q - row0, r_minus = r_plus + 1;
        const bool has_plus = r_plus >= 0, has_minus = r_minus < n_rows;
        es_perturb_float4<true>(theta, o, j4, sig, keys, tag, gen, (uint32_t)q,
                                has_plus ? out + r_plus * pitch : nullptr, has_minus ? out + r_minus * pitch : nullptr,
                                noise_out && has_plus ? noise_out + r_plus * pitch : nullptr,
                                noise_out && has_minus ? noise_out + r_minus * pitch : nullptr);
    }
}

// K5 for rows whose perturbable parameters are a PREFIX of the row: DeepQN rows hold the conv / Linear
// tensors first and the six BatchNorm vectors last (Atari/deepqn.py:158-172 get_perturbable_layers skips
// them), so parameter j is perturbed iff j < d_pert.
__global__ void __launch_bounds__(PT) es_perturb_prefix_kernel(
    const float* __restrict__ theta, int64_t d_pert, int64_t d_total, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0, float* __restrict__ out) {
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const int64_t r = blockIdx.x;
    const int64_t j4 = (int64_t)blockIdx.y * PT + threadIdx.x;
    if (j4 * 4 >= pitch) return;
    const float4 pv = *reinterpret_cast<const float4*>(theta + j4 * 4);
    float p[4] = {pv.x, pv.y, pv.z, pv.w};
    if (j4 * 4 < d_pert) {
        float z[4];
        normal4(keys, tag, gen, (uint32_t)(row0 + r), (uint32_t)j4, z);
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (j4 * 4 + i < d_pert) p[i] = __fadd_rn(p[i], __fmul_rn(sigma, z[i]));
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (j4 * 4 + i >= d_total) p[i] = 0.f;
    __stcs(reinterpret_cast<float4*>(out + r * pitch + j4 * 4), make_float4(p[0], p[1], p[2], p[3]));
}

// ---------------------------------------------------------------------------
// K6  ES update   (evolutionary_strategy.py:120-148)
// delta = lr/(n*sigma) * sum_i (sigma*z_i) * F_i, noise regenerated from the
// Philox key.  Members are split over blockIdx.y; partial sums are reduced in a
// fixed order by the second kernel (deterministic, no atomics).
// ---------------------------------------------------------------------------
// Partial sum over the local rows [r_lo, r_hi) of split `sp`, in row order.  MIRROR: member c = row0 + r carries
// s_c * (sigma z_q) with q = c >> 1, s_c = +1 for even c, -1 for odd c; z_q is generated once per pair, so the
// terms, and their order, are those of the per-member loop (the negation is exact).
//
// DIAG (separable NES): no sigma; two sums of the raw normals, sum_i F_i z_i into `partial` and
// sum_i F_i (z_i^2 - 1) into `partial_sigma` (the z^2 - 1 factor is fl(fl(z z) - 1); under mirroring (s z)^2 = z^2
// exactly, so both members of a pair add the same factor).
template <bool MIRROR, bool DIAG = false>
__device__ __forceinline__ void es_update_partial_body(
    const double* __restrict__ fitness, int in_dim, int64_t pitch, float sigma, const PhiloxKeys& keys,
    uint32_t tag, uint32_t gen, int64_t row0, int64_t r_lo, int64_t r_hi, int sp, float* __restrict__ partial,
    float* __restrict__ partial_sigma = nullptr) {
    const FcOffsets o = fc_offsets(in_dim);
    const int j4 = blockIdx.x * PT + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    float acc2[4] = {0.f, 0.f, 0.f, 0.f};
    bool pert[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int j = j4 * 4 + i;
        pert[i] = j < o.total && fc_is_perturbable(o, j);
    }
    if (pert[0] || pert[1] || pert[2] || pert[3]) {
        if (!MIRROR) {
            for (int64_t r = r_lo; r < r_hi; ++r) {
                const float f = (float)fitness[r];
                float z[4];
                normal4(keys, tag, gen, (uint32_t)(row0 + r), (uint32_t)j4, z);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (DIAG) {
                        acc[i] = fmaf(z[i], f, acc[i]);
                        acc2[i] = fmaf(__fsub_rn(__fmul_rn(z[i], z[i]), 1.f), f, acc2[i]);
                    } else {
                        acc[i] = fmaf(__fmul_rn(sigma, z[i]), f, acc[i]);
                    }
                }
            }
        } else {
            for (int64_t r = r_lo; r < r_hi;) {
                const int64_t c = row0 + r;
                float z[4], zz[4];
                normal4(keys, tag, gen, (uint32_t)(c >> 1), (uint32_t)j4, z);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (DIAG) zz[i] = __fsub_rn(__fmul_rn(z[i], z[i]), 1.f);
                    else z[i] = __fmul_rn(sigma, z[i]);
                }
                if (!(c & 1)) {
                    const float f = (float)fitness[r];
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        acc[i] = fmaf(z[i], f, acc[i]);
                        if (DIAG) acc2[i] = fmaf(zz[i], f, acc2[i]);
                    }
                    if (++r == r_hi) break;
                }
                const float f = (float)fitness[r];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    acc[i] = fmaf(-z[i], f, acc[i]);
                    if (DIAG) acc2[i] = fmaf(zz[i], f, acc2[i]);
                }
                ++r;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
        if (!pert[i]) acc[i] = acc2[i] = 0.f;
    *reinterpret_cast<float4*>(partial + (int64_t)sp * pitch + (int64_t)j4 * 4) =
        make_float4(acc[0], acc[1], acc[2], acc[3]);
    if (DIAG)
        *reinterpret_cast<float4*>(partial_sigma + (int64_t)sp * pitch + (int64_t)j4 * 4) =
            make_float4(acc2[0], acc2[1], acc2[2], acc2[3]);
}

// Local rows [r_lo, r_hi) of split sp.  Plain: n_split equal blocks of the local rows.  Mirrored sampling: the
// splits cover GLOBAL rows [base + sp*per, base + (sp+1)*per) of this rank's block, with base = row0 rounded down
// to even and `per` even, so every split but the first starts on a pair.
template <bool MIRROR>
__device__ __forceinline__ void es_update_split(int64_t row0, int64_t n_rows, int n_split, int sp, int64_t& r_lo,
                                                int64_t& r_hi) {
    if (!MIRROR) {
        const int64_t per = (n_rows + n_split - 1) / n_split;
        r_lo = sp * per;
        r_hi = min(n_rows, r_lo + per);
    } else {
        const int64_t base = row0 & ~(int64_t)1;
        const int64_t span = row0 + n_rows - base;
        const int64_t per = ((span + n_split - 1) / n_split + 1) & ~(int64_t)1;
        r_lo = max(base + sp * per, row0) - row0;
        r_hi = min(base + (sp + 1) * per, row0 + n_rows) - row0;
    }
}

__global__ void __launch_bounds__(PT) es_update_partial_kernel(
    const double* __restrict__ fitness, int in_dim, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows,
    int n_split, float* __restrict__ partial) {
    const int sp = blockIdx.y;
    int64_t r_lo, r_hi;
    es_update_split<false>(row0, n_rows, n_split, sp, r_lo, r_hi);
    es_update_partial_body<false>(fitness, in_dim, pitch, pick_sigma(sigma_arg, sigma_dev), keys, tag, gen, row0,
                                  r_lo, r_hi, sp, partial);
}

__global__ void __launch_bounds__(PT) es_update_mirrored_partial_kernel(
    const double* __restrict__ fitness, int in_dim, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev,
    const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows,
    int n_split, float* __restrict__ partial) {
    const int sp = blockIdx.y;
    int64_t r_lo, r_hi;
    es_update_split<true>(row0, n_rows, n_split, sp, r_lo, r_hi);
    es_update_partial_body<true>(fitness, in_dim, pitch, pick_sigma(sigma_arg, sigma_dev), keys, tag, gen, row0,
                                 r_lo, r_hi, sp, partial);
}

// K6 of separable NES, noise regenerated: partial sums of F_i z_i and F_i (z_i^2 - 1) over the splits of the plain /
// mirrored K6.  partial_sigma = partial + n_split * pitch.
template <bool MIRROR>
__global__ void __launch_bounds__(PT) es_update_diag_partial_kernel(
    const double* __restrict__ fitness, int in_dim, int64_t pitch, const PhiloxKeys keys, uint32_t tag, uint32_t gen,
    int64_t row0, int64_t n_rows, int n_split, float* __restrict__ partial) {
    const int sp = blockIdx.y;
    int64_t r_lo, r_hi;
    es_update_split<MIRROR>(row0, n_rows, n_split, sp, r_lo, r_hi);
    es_update_partial_body<MIRROR, true>(fitness, in_dim, pitch, 0.f, keys, tag, gen, row0, r_lo, r_hi, sp, partial,
                                         partial + (int64_t)n_split * pitch);
}

// g_mu = fl32(1/n_total) * (sum of the splits in order), g_sigma likewise from the second half of the workspace
__global__ void __launch_bounds__(PT) es_update_diag_finish_kernel(
    const float* __restrict__ partial, int n_split, int64_t pitch, double n_total, float* __restrict__ g_mu,
    float* __restrict__ g_sigma) {
    const int64_t j = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (j >= pitch) return;
    const float inv_n = (float)(1.0 / n_total);
    const float* partial_sigma = partial + (int64_t)n_split * pitch;
    float s = 0.f, t = 0.f;
    for (int sp = 0; sp < n_split; ++sp) {
        s += partial[(int64_t)sp * pitch + j];
        t += partial_sigma[(int64_t)sp * pitch + j];
    }
    g_mu[j] = __fmul_rn(inv_n, s);
    g_sigma[j] = __fmul_rn(inv_n, t);
}

// The same partial sums from the MATERIALISED members: sigma z_i = member_i - theta up to one rounding
// of the perturbation's add (1e-7 relative), read back at HBM speed instead of regenerating P normals per
// parameter on the ALU.  LayerNorm entries are copies of theta, so they contribute exact zeros.
__global__ void __launch_bounds__(PT) es_update_members_partial_kernel(
    const double* __restrict__ fitness, const float* __restrict__ members, const float* __restrict__ theta,
    int64_t pitch, int64_t n_rows, int n_split, float* __restrict__ partial) {
    const int j4 = blockIdx.x * PT + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    const int sp = blockIdx.y;
    const int64_t per = (n_rows + n_split - 1) / n_split;
    const int64_t r_lo = sp * per, r_hi = min(n_rows, r_lo + per);
    const float4 t4 = *reinterpret_cast<const float4*>(theta + (int64_t)j4 * 4);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float4* col = reinterpret_cast<const float4*>(members) + j4;
    const int64_t stride4 = pitch / 4;
#pragma unroll 8
    for (int64_t r = r_lo; r < r_hi; ++r) {
        const float f = (float)fitness[r];
        const float4 m = __ldcs(col + r * stride4);
        acc[0] = fmaf(__fsub_rn(m.x, t4.x), f, acc[0]);
        acc[1] = fmaf(__fsub_rn(m.y, t4.y), f, acc[1]);
        acc[2] = fmaf(__fsub_rn(m.z, t4.z), f, acc[2]);
        acc[3] = fmaf(__fsub_rn(m.w, t4.w), f, acc[3]);
    }
    *reinterpret_cast<float4*>(partial + (int64_t)sp * pitch + (int64_t)j4 * 4) =
        make_float4(acc[0], acc[1], acc[2], acc[3]);
}

// coefficient lr / (n_total * sigma) in fp64 like the reference's Python float, then one fp32 multiply
__global__ void __launch_bounds__(PT) es_update_finish_kernel(
    const float* __restrict__ partial, int n_split, int64_t pitch, double lr, double n_total, float sigma_arg,
    const double* __restrict__ sigma_dev, float* __restrict__ delta) {
    const int64_t j = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (j >= pitch) return;
    const float coef = (float)(lr / (n_total * (double)pick_sigma(sigma_arg, sigma_dev)));
    float s = 0.f;
    for (int sp = 0; sp < n_split; ++sp) s += partial[(int64_t)sp * pitch + j];
    delta[j] = __fmul_rn(coef, s);
}

__global__ void __launch_bounds__(PT) axpy_kernel(float a, const float* __restrict__ x,
                                                  float* __restrict__ y, int64_t n) {
    const int64_t j = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (j < n) y[j] = __fadd_rn(y[j], __fmul_rn(a, x[j]));
}

// ---------------------------------------------------------------------------
// Centered-rank fitness shaping (Salimans et al. 2017; extends evolutionary_strategy.py:120-148, whose
// normalisation is commented out at :133-135).  u_i = r_i / (P-1) - 0.5 with the average rank
// r_i = #{F_j < F_i} + (#{F_j == F_i} - 1) / 2 over the GLOBAL fitness; the thread of local row r ranks member
// row0 + r against all P keys staged in shared-memory tiles (integer compares only: P * n_rows of them).
// ---------------------------------------------------------------------------
constexpr int RK_T = 256;
constexpr int RK_TILE = 2048;          // keys per tile: 16 KB of shared memory

// Order-preserving key of an fp64 value: -0.0 maps to +0.0's key, every NaN to 0 (below -inf, whose key is
// 0x000FFFFFFFFFFFFF): all NaNs tie and rank below every number.
__device__ __forceinline__ unsigned long long rank_key(double x) {
    if (x != x) return 0ull;
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    if ((b << 1) == 0ull) b = 0ull;
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

__global__ void __launch_bounds__(RK_T) centered_ranks_kernel(const double* __restrict__ fitness, int64_t P,
                                                              int64_t row0, int64_t n_rows,
                                                              double* __restrict__ out) {
    __shared__ unsigned long long tile[RK_TILE];
    const int64_t r = (int64_t)blockIdx.x * RK_T + threadIdx.x;
    const unsigned long long k = r < n_rows ? rank_key(fitness[row0 + r]) : 0ull;
    int64_t lt = 0, eq = 0;
    for (int64_t t0 = 0; t0 < P; t0 += RK_TILE) {
        const int n = (int)min((int64_t)RK_TILE, P - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < n; i += RK_T) tile[i] = rank_key(fitness[t0 + i]);
        __syncthreads();
        int lt_t = 0, eq_t = 0;
#pragma unroll 8
        for (int i = 0; i < n; ++i) {
            const unsigned long long kj = tile[i];
            lt_t += kj < k;
            eq_t += kj == k;
        }
        lt += lt_t;
        eq += eq_t;
    }
    if (r >= n_rows) return;
    const double rank = __dadd_rn((double)lt, __dmul_rn(0.5, (double)(eq - 1)));   // exact: a multiple of 1/2
    out[r] = P > 1 ? __dsub_rn(__ddiv_rn(rank, (double)(P - 1)), 0.5) : 0.0;
}

// ---------------------------------------------------------------------------
// Fused ES apply over the roles' concatenated rows (extends evolutionary_strategy.py:259-265; the reference
// builds an Adam optimizer per agent and never uses it, MPE/mpe_agent.py:20).  g = ghat - l2 * theta, then
//   sgd:  theta += lr * g
//   adam: m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g g ; theta += alpha_t m / (sqrt(v) + eps)
// one IEEE-rounded fp32 operation at a time (no contraction), on the perturbable entries only: LayerNorm
// entries and padding of theta, m and v keep their bits.
// ---------------------------------------------------------------------------
struct ApplySegments {
    int n;
    int in_dim[CEV_MAX_ROLES];
    int64_t end[CEV_MAX_ROLES];        // exclusive end offset of each segment in the concatenated row
};

__global__ void __launch_bounds__(PT) es_apply_kernel(float* __restrict__ theta, const float* __restrict__ delta,
                                                      float* __restrict__ m, float* __restrict__ v,
                                                      const ApplySegments seg, int adam, float step, float l2) {
    const int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x;
    int in_dim = seg.in_dim[0];
    int64_t start = 0, end = seg.end[0];
#pragma unroll
    for (int s = 1; s < CEV_MAX_ROLES; ++s)          // constant indices: the segment table stays in registers
        if (s < seg.n && i >= end) { in_dim = seg.in_dim[s]; start = end; end = seg.end[s]; }
    if (i >= end) return;
    const FcOffsets o = fc_offsets(in_dim);
    const int j = (int)(i - start);
    if (j >= o.total || !fc_is_perturbable(o, j)) return;
    const float th = theta[i];
    const float g = __fsub_rn(delta[i], __fmul_rn(l2, th));
    if (!adam) {
        theta[i] = __fadd_rn(th, __fmul_rn(step, g));
        return;
    }
    const float b1 = CEV_ADAM_BETA1, b2 = CEV_ADAM_BETA2, eps = CEV_ADAM_EPS;
    const float mi = __fadd_rn(__fmul_rn(b1, m[i]), __fmul_rn(__fsub_rn(1.f, b1), g));
    const float vi = __fadd_rn(__fmul_rn(b2, v[i]), __fmul_rn(__fmul_rn(__fsub_rn(1.f, b2), g), g));
    m[i] = mi;
    v[i] = vi;
    theta[i] = __fadd_rn(th, __fdiv_rn(__fmul_rn(step, mi), __fadd_rn(__fsqrt_rn(vi), eps)));
}

// Separable NES apply (Wierstra et al. 2014, SNES) over the same concatenated rows, perturbable entries only:
//   theta += fl(lr * fl(sigma * g_mu))                          (the old sigma)
//   sigma  = clamp(fl(sigma * fl32(exp(half_eta[s] * g_sigma))), sigma_min, sigma_max)     (exp in fp64)
// half_eta[s] = eta_sigma / 2 of segment s.  fminf / fmaxf: a NaN product clamps to sigma_min.
struct DiagEta {
    double half[CEV_MAX_ROLES];
};

__global__ void __launch_bounds__(PT) es_apply_diag_kernel(float* __restrict__ theta, float* __restrict__ sigma,
                                                           const float* __restrict__ g_mu,
                                                           const float* __restrict__ g_sigma, const ApplySegments seg,
                                                           const DiagEta eta, float lr, float sigma_min,
                                                           float sigma_max) {
    const int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x;
    int in_dim = seg.in_dim[0];
    double half_eta = eta.half[0];
    int64_t start = 0, end = seg.end[0];
#pragma unroll
    for (int s = 1; s < CEV_MAX_ROLES; ++s)          // constant indices: the tables stay in registers
        if (s < seg.n && i >= end) { in_dim = seg.in_dim[s]; half_eta = eta.half[s]; start = end; end = seg.end[s]; }
    if (i >= end) return;
    const FcOffsets o = fc_offsets(in_dim);
    const int j = (int)(i - start);
    if (j >= o.total || !fc_is_perturbable(o, j)) return;
    const float s = sigma[i];
    theta[i] = __fadd_rn(theta[i], __fmul_rn(lr, __fmul_rn(s, g_mu[i])));
    const float factor = (float)exp(__dmul_rn(half_eta, (double)g_sigma[i]));
    sigma[i] = fminf(fmaxf(__fmul_rn(s, factor), sigma_min), sigma_max);
}

// ---------------------------------------------------------------------------
// K7  fitness-sharing distances   (utils/game_logic_functions.py:12-21)
// d[i] = || pop[i] - ref ||_2 over the Linear parameters; one CTA per row.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(PT) diversity_dist_kernel(
    const float* __restrict__ pop, int64_t pitch, const float* __restrict__ ref, int in_dim,
    float* __restrict__ dist) {
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r = blockIdx.x;
    const float4* row = reinterpret_cast<const float4*>(pop + r * pitch);
    const float4* rf = reinterpret_cast<const float4*>(ref);
    float acc = 0.f;
    // every segment boundary is a multiple of 4 parameters except the end of the row: a float4 is
    // perturbable or not as a whole; four independent 128-bit loads in flight per thread
    const int n4 = (int)(pitch / 4);
#pragma unroll 4
    for (int j4 = threadIdx.x; j4 < n4; j4 += PT) {
        const int j = j4 * 4;
        if (j >= o.total || !fc_is_perturbable(o, j)) continue;
        const float4 a = __ldcs(row + j4);
        const float4 b = __ldg(rf + j4);
        const float d[4] = {a.x - b.x, a.y - b.y, a.z - b.z, a.w - b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (j + i < o.total) acc = fmaf(d[i], d[i], acc);
    }
    __shared__ float red[PT / 32];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < PT / 32; ++w) s += red[w];
        dist[r] = sqrtf(s);
    }
}

// ---------------------------------------------------------------------------
// K4  selection   (genetic_algorithm.py:223-234)
// k rounds of a block-wide arg-max over the not-yet-chosen members (a byte mask in the workspace, so
// k is unbounded).  Two total orders:
//   order 0: value descending, ties -> LOWER index, NaN ranks last  (= argsort(-f, kind="stable"))
//   order 1: the reference's expression np.argsort(f)[::-1] with a stable ascending sort (what
//            NumPy's small-array insertion sort does): value descending, ties -> HIGHER index, NaN
//            ranks FIRST (Appendix C #18).
// Single CTA: P <= a few 1e5 and a handful of elites is latency-bound.
// ---------------------------------------------------------------------------
constexpr int SEL_T = 1024;

__device__ __forceinline__ bool sel_better(double va, int64_t ia, double vb, int64_t ib, int order) {
    // is (va, ia) ranked before (vb, ib)?
    if (ib < 0) return ia >= 0;
    if (ia < 0) return false;
    const bool na = va != va, nb = vb != vb;
    if (na || nb) {
        if (na != nb) return order ? na : nb;            // order 1: NaN first; order 0: NaN last
        return order ? ia > ib : ia < ib;
    }
    if (va > vb) return true;
    if (va < vb) return false;
    return order ? ia > ib : ia < ib;
}

__global__ void __launch_bounds__(SEL_T) select_topk_kernel(const double* __restrict__ fitness, int64_t P,
                                                            int k, int order, uint8_t* __restrict__ taken,
                                                            int64_t* __restrict__ idx_out) {
    __shared__ double wv[SEL_T / 32];
    __shared__ int64_t wi[SEL_T / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int64_t i = threadIdx.x; i < P; i += SEL_T) taken[i] = 0;
    __syncthreads();
    for (int round = 0; round < k; ++round) {
        double bv = 0.0;
        int64_t bi = -1;
        for (int64_t i = threadIdx.x; i < P; i += SEL_T) {
            if (taken[i]) continue;
            const double v = fitness[i];
            if (sel_better(v, i, bv, bi, order)) { bv = v; bi = i; }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const double ov = __shfl_xor_sync(0xffffffffu, bv, off);
            const int64_t oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (sel_better(ov, oi, bv, bi, order)) { bv = ov; bi = oi; }
        }
        if (lane == 0) { wv[warp] = bv; wi[warp] = bi; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double v = wv[0];
            int64_t ix = wi[0];
            for (int w = 1; w < SEL_T / 32; ++w)
                if (sel_better(wv[w], wi[w], v, ix, order)) { v = wv[w]; ix = wi[w]; }
            taken[ix] = 1;
            idx_out[round] = ix;
        }
        __syncthreads();
    }
}

// dst[r] = src[idx[r] - row0] when the GLOBAL row id idx[r] lies in this rank's block
// [row0, row0 + n_local), zeros otherwise: summed over ranks (all-reduce) the result is the
// elite / Hall-of-Fame broadcast with no host round trip for the indices.  n_local < 0: no range
// (plain gather of local ids).
__global__ void __launch_bounds__(PT) gather_rows_kernel(const float* __restrict__ src, int64_t pitch,
                                                         const int64_t* __restrict__ idx, int64_t row0,
                                                         int64_t n_local, float* __restrict__ dst) {
    const int64_t r = blockIdx.x;
    const int64_t s = idx[r] - row0;
    const int j4 = blockIdx.y * PT + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (n_local < 0 || (s >= 0 && s < n_local)) v = *reinterpret_cast<const float4*>(src + s * pitch + (int64_t)j4 * 4);
    *reinterpret_cast<float4*>(dst + r * pitch + (int64_t)j4 * 4) = v;
}

// ---------------------------------------------------------------------------
// Per-member statistics of the perturbable weights (MPEAgent.log_weight_statistics,
// MPE/mpe_agent.py:30-50: mean, min, max, population std of get_perturbable_weights()).
// One CTA per row, HBM-read bound (4 B/param/member); out fp32 [n_rows][4] = mean, min, max, std.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(PT) weight_stats_kernel(const float* __restrict__ rows, int64_t pitch, int in_dim,
                                                          float* __restrict__ out) {
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r = blockIdx.x;
    const float* row = rows + r * pitch;
    double sum = 0.0, sq = 0.0;
    float mn = CUDART_INF_F, mx = -CUDART_INF_F;
    const int n4 = (int)(pitch / 4);
#pragma unroll 4
    for (int j4 = threadIdx.x; j4 < n4; j4 += PT) {
        const int j = j4 * 4;
        if (j >= o.total || !fc_is_perturbable(o, j)) continue;
        const float4 a = __ldcs(reinterpret_cast<const float4*>(row) + j4);
        const float v[4] = {a.x, a.y, a.z, a.w};
        // fp32 partial sums of one float4, fp64 across float4s (138 k terms per row)
        float s4 = 0.f, q4 = 0.f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (j + i < o.total) {
                s4 += v[i];
                q4 = fmaf(v[i], v[i], q4);
                mn = fminf(mn, v[i]);
                mx = fmaxf(mx, v[i]);
            }
        }
        sum += (double)s4;
        sq += (double)q4;
    }
    __shared__ double rs[PT / 32], rq[PT / 32];
    __shared__ float rmn[PT / 32], rmx[PT / 32];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, off);
        sq += __shfl_xor_sync(0xffffffffu, sq, off);
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
    }
    if ((threadIdx.x & 31) == 0) {
        rs[threadIdx.x >> 5] = sum; rq[threadIdx.x >> 5] = sq;
        rmn[threadIdx.x >> 5] = mn; rmx[threadIdx.x >> 5] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < PT / 32; ++w) {
            sum += rs[w]; sq += rq[w];
            mn = fminf(mn, rmn[w]); mx = fmaxf(mx, rmx[w]);
        }
        const double n = (double)(o.total - 2 * (H1 + H2));
        const double mean = sum / n;
        const double var = fmax(sq / n - mean * mean, 0.0);
        float4 res = make_float4((float)mean, mn, mx, (float)sqrt(var));
        *reinterpret_cast<float4*>(out + r * 4) = res;
    }
}

// ---------------------------------------------------------------------------
// End of a generation, on the device (SURVEY.md 8f N1): the mean reward triple of the evaluation
// games (evaluate_current_weights, genetic_algorithm.py:12-29 == evolutionary_strategy.py:22-59),
// the reward history, the adaptive mutation power (genetic_algorithm.py:323-345 ==
// evolutionary_strategy.py:292-316, including agent_0 growing from sigma_agent_1 * 1.2, Appendix C #6)
// and the early-stopping counters (evolutionary_strategy.py:318-354).  One thread: it is ~100 scalar
// operations, and what matters is that nothing leaves the device between generations.
// gstate (fp64) layout: see CEV_GS_* in the header.
// ---------------------------------------------------------------------------
// NumPy's pairwise summation for n < 128 (np.mean of a list of Python floats): eight running sums
// for n >= 8, a plain loop below that.
__device__ double np_mean(const double* a, int n) {
    if (n <= 0) return CUDART_NAN;
    double res;
    if (n < 8) {
        res = 0.0;
        for (int i = 0; i < n; ++i) res += a[i];
    } else {
        double r[8];
        for (int j = 0; j < 8; ++j) r[j] = a[j];
        int i = 8;
        for (; i < n - (n % 8); i += 8)
            for (int j = 0; j < 8; ++j) r[j] += a[i + j];
        res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; ++i) res += a[i];
    }
    return res / (double)n;
}

__global__ void generation_end_kernel(const double* __restrict__ eval_out, int n_games, int agent_step_limit,
                                      int reference_compat, double* __restrict__ gs, int hist_cap, int adaptive,
                                      double sigma_max, double sigma_min, int early_stopping, double min_delta,
                                      int patience) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int gen = (int)gs[CEV_GS_GEN];
    // ---- reward slots of play_MPE (utils/game_logic_functions.py:179-190, Appendix B) ----------
    const int L = agent_step_limit < 0 ? 75 : min(75, max(0, agent_step_limit));
    const int nc = L / 3;
    const int n_adv = (L + 2) / 3, n_a0 = (L + 1) / 3;     // ceil(L/3), ceil((L-1)/3) for L >= 1
    double tot[3] = {0.0, 0.0, 0.0};
    for (int g = 0; g < n_games; ++g) {
        const double sg = eval_out[g * CEV_ROLLOUT_OUT_DIM + 0], lg = eval_out[g * CEV_ROLLOUT_OUT_DIM + 1],
                     sa = eval_out[g * CEV_ROLLOUT_OUT_DIM + 2];
        double s0, s1, sadv;
        if (!reference_compat) { s0 = sg; s1 = sg; sadv = sa; }
        else if (nc == 0) { s0 = 0.0; s1 = sa; sadv = 0.0; }
        else {
            sadv = (n_adv - 1 >= nc) ? sg : sg - lg;
            s0 = (n_a0 - 1 >= nc) ? sg : sg - lg;
            s1 = sa;
        }
        tot[0] += s0; tot[1] += s1; tot[2] += sadv;       // the reference's running sums, game order
    }
    double ev[3];
    for (int r = 0; r < 3; ++r) ev[r] = tot[r] / (double)n_games;
    double* hist = gs + CEV_GS_HIST;                      // [hist_cap][3]
    double* shist = hist + (size_t)3 * hist_cap;          // [hist_cap + 1][3], entry 0 = initial sigma
    if (gen < hist_cap)
        for (int r = 0; r < 3; ++r) hist[(size_t)gen * 3 + r] = ev[r];
    for (int r = 0; r < 3; ++r) gs[CEV_GS_LAST_EVAL + r] = ev[r];
    // ---- adaptive mutation power ------------------------------------------------------------------
    if (adaptive) {
        double sig[3] = {gs[CEV_GS_SIGMA + 0], gs[CEV_GS_SIGMA + 1], gs[CEV_GS_SIGMA + 2]};
        const int n = gen + 1;                            // rewards recorded so far
        for (int r = 0; r < 3; ++r) {
            bool worse = false;
            if (gen > 10 && n <= hist_cap) {
                // lists sliced like Python: h[-10:] and h[-20:-10]
                double last[10], prev[10];
                const int n_last = min(n, 10);
                for (int i = 0; i < n_last; ++i) last[i] = hist[(size_t)(n - n_last + i) * 3 + r];
                const int lo = max(0, n - 20), hi = max(0, n - 10);
                const int n_prev = hi - lo;
                for (int i = 0; i < n_prev; ++i) prev[i] = hist[(size_t)(lo + i) * 3 + r];
                worse = np_mean(last, n_last) < np_mean(prev, n_prev);
            }
            // agent_0 (r = 0) grows from sigma_agent_1 (already this generation's old value: agent_0 is
            // updated first), Appendix C #6
            if (worse) sig[r] = fmin((r == 0 ? sig[1] : sig[r]) * 1.2, sigma_max);
            else sig[r] = fmax(sig[r] * 0.95, sigma_min);
        }
        for (int r = 0; r < 3; ++r) gs[CEV_GS_SIGMA + r] = sig[r];
    }
    if (gen + 1 <= hist_cap)
        for (int r = 0; r < 3; ++r) shist[(size_t)(gen + 1) * 3 + r] = gs[CEV_GS_SIGMA + r];
    // ---- early stopping ---------------------------------------------------------------------------
    if (early_stopping && gs[CEV_GS_STOP] == 0.0) {
        for (int r = 0; r < 3; ++r) {
            if (ev[r] > gs[CEV_GS_BEST + r] + min_delta) {
                gs[CEV_GS_BEST + r] = ev[r];
                gs[CEV_GS_STALE + r] = 0.0;
            } else {
                gs[CEV_GS_STALE + r] += 1.0;
            }
        }
        for (int r = 0; r < 3; ++r)
            if (gs[CEV_GS_STALE + r] >= (double)patience) {
                gs[CEV_GS_STOP] = (double)(1 + r);        // first role in agent_0, agent_1, adversary order
                gs[CEV_GS_STOP_GEN] = (double)gen;
                break;
            }
    }
    gs[CEV_GS_GEN] = (double)(gen + 1);
}

// ---------------------------------------------------------------------------
// synthetic inputs
// ---------------------------------------------------------------------------
__device__ __forceinline__ double u_pm1(uint32_t x) {
    // uniform in (-1, 1): ((x + 0.5) * 2^-32) * 2 - 1, exact in fp64
    return ((double)x + 0.5) * (2.0 / 4294967296.0) - 1.0;
}

__global__ void __launch_bounds__(PT) init_states_kernel(uint32_t k0, uint32_t k1, uint32_t stream_id,
                                                         int64_t rec0, int64_t n, double* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (i >= n) return;
    const int64_t r = rec0 + i;
    const uint32_t tag = noise_tag(CEV_KIND_ENV, 0);
    uint32_t w[12];
#pragma unroll
    for (int b = 0; b < 3; ++b) {
        const U4 v = philox4x32_10(U4{(uint32_t)b, (uint32_t)r, stream_id, tag}, k0, k1);
        w[4 * b] = v.x; w[4 * b + 1] = v.y; w[4 * b + 2] = v.z; w[4 * b + 3] = v.w;
    }
    double* o = out + i * CEV_INIT_STATE_DIM;
    o[0] = (double)(w[0] & 1u);
#pragma unroll
    for (int i = 0; i < 10; ++i) o[1 + i] = u_pm1(w[1 + i]);
}

// Founder initialisation on the device (create_agent -> FCNetwork default init,
// MPE/fcnetwork.py:11-22): nn.Linear weight and bias ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)),
// LayerNorm gamma = 1, beta = 0.  Same distribution as PyTorch's default, Philox stream
// (kind 4) instead of torch's global generator; needed when P is too large to build
// 3*P nn.Modules on the host.
__global__ void __launch_bounds__(PT) fc_init_kernel(int in_dim, int64_t pitch, uint32_t k0, uint32_t k1,
                                                     uint32_t tag, int64_t row0, float* __restrict__ out) {
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r = blockIdx.x;
    const int j4 = blockIdx.y * PT + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    const U4 w = philox4x32_10(U4{(uint32_t)j4, (uint32_t)(row0 + r), 0u, tag}, k0, k1);
    const uint32_t x[4] = {w.x, w.y, w.z, w.w};
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int j = j4 * 4 + i;
        if (j >= o.total) v[i] = 0.f;
        else if (j >= o.ln1g && j < o.ln1b) v[i] = 1.f;
        else if (j >= o.ln1b && j < o.fc2w) v[i] = 0.f;
        else if (j >= o.ln2g && j < o.ln2b) v[i] = 1.f;
        else if (j >= o.ln2b && j < o.outw) v[i] = 0.f;
        else {
            const int fan_in = j < o.ln1g ? in_dim : (j < o.ln2g ? H1 : H2);
            const double bound = 1.0 / sqrt((double)fan_in);
            const double u = ((double)x[i] + 0.5) * (2.0 / 4294967296.0) - 1.0;
            v[i] = (float)(u * bound);
        }
    }
    *reinterpret_cast<float4*>(out + r * pitch + (int64_t)j4 * 4) = make_float4(v[0], v[1], v[2], v[3]);
}

__global__ void __launch_bounds__(PT) random_frames_kernel(uint32_t k0, uint32_t k1, int64_t n16,
                                                           uint4* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (i >= n16) return;
    const U4 v = philox4x32_10(U4{(uint32_t)i, (uint32_t)(i >> 32), 0u, noise_tag(CEV_KIND_FRAMES, 0)}, k0, k1);
    out[i] = make_uint4(v.x, v.y, v.z, v.w);
}

__global__ void __launch_bounds__(PT) philox_words_kernel(uint32_t k0, uint32_t k1, uint32_t tag, uint32_t gen,
                                                          int64_t member0, int64_t n_members, int64_t n4,
                                                          uint4* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * PT + threadIdx.x;
    if (i >= n_members * n4) return;
    const int64_t m = i / n4, j4 = i % n4;
    const U4 v = philox4x32_10(U4{(uint32_t)j4, (uint32_t)(member0 + m), gen, tag}, k0, k1);
    out[i] = make_uint4(v.x, v.y, v.z, v.w);
}

// Co-ES Hall of Fame: slot of opponent set k (0 = the newest snapshot, k >= 1 uniform over the filled slots)
__global__ void __launch_bounds__(PT) es_hof_opponents_kernel(uint32_t k0, uint32_t k1, uint32_t gen, int K,
                                                              uint64_t filled, int64_t newest,
                                                              int64_t* __restrict__ out) {
    const int k = blockIdx.x * PT + threadIdx.x;
    if (k >= K) return;
    if (k == 0) {
        out[0] = newest;
        return;
    }
    const U4 v = philox4x32_10(U4{(uint32_t)((k - 1) >> 2), 0u, gen, noise_tag(CEV_KIND_HOF, 0)}, k0, k1);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    out[k] = (int64_t)(((uint64_t)w[(k - 1) & 3] * filled) >> 32);
}

// ---------------------------------------------------------------------------
// FP32 FMA-pipe peak (roofline denominator for K1, SURVEY.md section 8d)
// ---------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters) {
    float2 a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = make_float2(threadIdx.x * 1e-3f + i, blockIdx.x * 1e-3f - i);
    const float2 b = make_float2(0.999f, 1.001f), c = make_float2(1e-3f, -1e-3f);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (MODE == 1) a[i] = __ffma2_rn(a[i], b, c);
            else { a[i].x = fmaf(a[i].x, b.x, c.x); a[i].y = fmaf(a[i].y, b.y, c.y); }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += a[i].x + a[i].y;
    if (s == 123.456f) out[0] = s;       // keep the chain alive
}

}  // namespace cev

using namespace cev;

static inline void split_seed(uint64_t seed, uint32_t& k0, uint32_t& k1) {
    k0 = (uint32_t)(seed & 0xFFFFFFFFull);
    k1 = (uint32_t)(seed >> 32);
}

static int ensure_workspace(cev_handle* h, size_t bytes) {
    if (h->workspace_bytes >= bytes) return CEV_OK;
    if (h->workspace) cudaFree(h->workspace);
    h->workspace = nullptr;
    h->workspace_bytes = 0;
    CEV_CUDA(cudaMalloc(&h->workspace, bytes));
    h->workspace_bytes = bytes;
    return CEV_OK;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

int cev_ga_repopulate_f32(cev_handle* h, const float* elites, int E, int D, int64_t pitch, float sigma,
                          const double* sigma_dev, float crossover_rate, uint64_t seed, int role, uint32_t gen,
                          int64_t row0, int64_t n_rows, float* out, float* noise_out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "ga_repopulate: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(elites && out, "ga_repopulate: null pointer");
    CEV_REQUIRE(E >= 1 && D >= 1 && pitch >= D && pitch % 4 == 0, "ga_repopulate: bad E/D/pitch");
    CEV_REQUIRE(crossover_rate >= 0.f && crossover_rate <= 1.f, "ga_repopulate: crossover_rate must be in [0, 1]");
    CEV_REQUIRE(aligned16(elites) && aligned16(out) && aligned16(noise_out), "ga_repopulate: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "ga_repopulate: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    dim3 grid((unsigned)n_rows, (unsigned)((pitch / 4 + PT - 1) / PT));
    ga_repopulate_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(elites, E, D, pitch, sigma, sigma_dev, philox_keys(k0, k1),
                                                               noise_tag(CEV_KIND_GA, role), gen, row0, crossover_rate,
                                                               noise_tag(CEV_KIND_XOVER, role), out, noise_out);
    return check_cuda(cudaGetLastError(), "ga_repopulate_kernel");
}

int cev_gather_rows_f32(cev_handle* h, const float* src, int64_t pitch, const int64_t* idx, int n, int64_t row0,
                        int64_t n_local, float* dst, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "gather_rows: null handle");
    if (n <= 0) return CEV_OK;
    // an empty shard (n_local == 0) has no rows to read: src may be null, dst is zero-filled
    CEV_REQUIRE((src || n_local == 0) && idx && dst, "gather_rows: null pointer");
    CEV_REQUIRE(pitch % 4 == 0 && aligned16(src) && aligned16(dst), "gather_rows: alignment");
    CEV_GUARD(h);
    dim3 grid((unsigned)n, (unsigned)((pitch / 4 + PT - 1) / PT));
    gather_rows_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(src, pitch, idx, row0, n_local, dst);
    return check_cuda(cudaGetLastError(), "gather_rows_kernel");
}

int cev_select_topk_f64(cev_handle* h, const double* fitness, int64_t P, int k, int order, int64_t* idx_out,
                        cev_stream stream) {
    CEV_REQUIRE(h && fitness && idx_out, "select_topk: null pointer");
    CEV_REQUIRE(k >= 1 && k <= P, "select_topk: need 1 <= k <= P (elites_number %d, population %lld)", k, (long long)P);
    CEV_REQUIRE(order == 0 || order == 1, "select_topk: order must be 0 (ties -> lower index) or 1 (reference)");
    CEV_GUARD(h);
    int rc = ensure_workspace(h, (size_t)P + 256);
    if (rc) return rc;
    select_topk_kernel<<<1, SEL_T, 0, (cudaStream_t)stream>>>(fitness, P, k, order, static_cast<uint8_t*>(h->workspace),
                                                              idx_out);
    return check_cuda(cudaGetLastError(), "select_topk_kernel");
}

int cev_es_perturb_f32(cev_handle* h, const float* theta, int in_dim, float sigma, const double* sigma_dev,
                       uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                       float* out, float* noise_out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(theta && out, "es_perturb: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_perturb: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "es_perturb: bad pitch");
    CEV_REQUIRE(aligned16(theta) && aligned16(out) && aligned16(noise_out), "es_perturb: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    dim3 grid((unsigned)n_rows, (unsigned)((pitch / 4 + K5T - 1) / K5T));
    es_perturb_kernel<<<grid, K5T, 0, (cudaStream_t)stream>>>(theta, in_dim, pitch, sigma, sigma_dev, philox_keys(k0, k1),
                                                            noise_tag(CEV_KIND_ES, role), gen, row0, out,
                                                            noise_out);
    return check_cuda(cudaGetLastError(), "es_perturb_kernel");
}

int cev_es_update_f32(cev_handle* h, const double* fitness, int in_dim, float sigma, const double* sigma_dev,
                      float lr, int64_t n_total, uint64_t seed, int role, uint32_t gen, int64_t row0,
                      int64_t n_rows, float* delta, cev_stream stream) {
    // an empty shard (n_rows == 0, fitness may be null) still writes its all-zero partial delta
    CEV_REQUIRE(h && (fitness || n_rows == 0) && delta, "es_update: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_update: in_dim must be 8 or 10");
    CEV_REQUIRE(n_total >= 1 && n_rows >= 0 && (sigma_dev || sigma > 0.f), "es_update: bad n/sigma");
    CEV_REQUIRE(aligned16(delta), "es_update: 16B alignment");
    CEV_GUARD(h);
    const int64_t pitch = fc_pitch(in_dim);
    int n_split = (int)((n_rows + 63) / 64);
    if (n_split > 16) n_split = 16;
    if (n_split < 1) n_split = 1;
    int rc = ensure_workspace(h, (size_t)n_split * pitch * sizeof(float));
    if (rc) return rc;
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    float* partial = static_cast<float*>(h->workspace);
    dim3 grid((unsigned)((pitch / 4 + PT - 1) / PT), (unsigned)n_split);
    es_update_partial_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(fitness, in_dim, pitch, sigma, sigma_dev, philox_keys(k0, k1),
                                                                   noise_tag(CEV_KIND_ES, role), gen, row0,
                                                                   n_rows, n_split, partial);
    CEV_CUDA(cudaGetLastError());
    es_update_finish_kernel<<<(unsigned)((pitch + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        partial, n_split, pitch, (double)lr, (double)n_total, sigma, sigma_dev, delta);
    return check_cuda(cudaGetLastError(), "es_update kernels");
}

int cev_es_perturb_prefix_f32(cev_handle* h, const float* theta, int64_t d_pert, int64_t d_total, float sigma,
                              const double* sigma_dev, uint64_t seed, int role, uint32_t gen, int64_t row0,
                              int64_t n_rows, int64_t pitch, float* out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb_prefix: null handle");
    if (n_rows == 0) return CEV_OK;
    CEV_REQUIRE(theta && out, "es_perturb_prefix: null pointer");
    CEV_REQUIRE(d_pert >= 0 && d_pert <= d_total && d_total <= pitch && pitch % 4 == 0 && pitch / 4 <= 0xFFFFFFFFll,
                "es_perturb_prefix: need 0 <= d_pert <= d_total <= pitch, pitch a multiple of 4");
    CEV_REQUIRE(aligned16(theta) && aligned16(out), "es_perturb_prefix: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb_prefix: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    dim3 grid((unsigned)n_rows, (unsigned)((pitch / 4 + PT - 1) / PT));
    es_perturb_prefix_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(theta, d_pert, d_total, pitch, sigma, sigma_dev, philox_keys(k0, k1),
                                                                   noise_tag(CEV_KIND_ES, role), gen, row0, out);
    return check_cuda(cudaGetLastError(), "es_perturb_prefix_kernel");
}

int cev_es_update_members_f32(cev_handle* h, const double* fitness, const float* members, int64_t pitch,
                              const float* theta, int in_dim, float sigma, const double* sigma_dev, float lr,
                              int64_t n_total, int64_t n_rows, float* delta, cev_stream stream) {
    // an empty shard (n_rows == 0: fitness / members may be null) still writes its all-zero partial delta
    CEV_REQUIRE(h && ((fitness && members) || n_rows == 0) && theta && delta, "es_update_members: null pointer");
    CEV_REQUIRE(n_total >= 1 && n_rows >= 0 && (sigma_dev || sigma > 0.f), "es_update_members: bad n/sigma");
    // in_dim 8 / 10: FCNetwork rows (pitch checked); in_dim 0: any row layout of `pitch` floats (DeepQN):
    // the kernel is layout agnostic, unperturbed entries are copies of theta and contribute exact zeros
    CEV_REQUIRE(in_dim == 0 || in_dim == IN_ADV || in_dim == IN_GOOD, "es_update_members: in_dim must be 0, 8 or 10");
    CEV_REQUIRE(in_dim == 0 ? (pitch > 0 && pitch % 4 == 0) : pitch == fc_pitch(in_dim),
                "es_update_members: rows must use the padded pitch (cev_fc_pitch / cev_dqn_pitch)");
    CEV_REQUIRE(aligned16(delta) && aligned16(members) && aligned16(theta), "es_update_members: 16B alignment");
    CEV_GUARD(h);
    int n_split = (int)((n_rows + 31) / 32);
    if (n_split > 32) n_split = 32;
    if (n_split < 1) n_split = 1;
    int rc = ensure_workspace(h, (size_t)n_split * pitch * sizeof(float));
    if (rc) return rc;
    float* partial = static_cast<float*>(h->workspace);
    dim3 grid((unsigned)((pitch / 4 + PT - 1) / PT), (unsigned)n_split);
    es_update_members_partial_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(fitness, members, theta, pitch, n_rows,
                                                                           n_split, partial);
    CEV_CUDA(cudaGetLastError());
    es_update_finish_kernel<<<(unsigned)((pitch + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        partial, n_split, pitch, (double)lr, (double)n_total, sigma, sigma_dev, delta);
    return check_cuda(cudaGetLastError(), "es_update_members kernels");
}

int cev_es_perturb_mirrored_f32(cev_handle* h, const float* theta, int in_dim, float sigma, const double* sigma_dev,
                                uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                                float* out, float* noise_out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb_mirrored: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(theta && out, "es_perturb_mirrored: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_perturb_mirrored: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "es_perturb_mirrored: bad pitch");
    CEV_REQUIRE(aligned16(theta) && aligned16(out) && aligned16(noise_out), "es_perturb_mirrored: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb_mirrored: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    const int64_t n_pairs = ((row0 + n_rows - 1) >> 1) - (row0 >> 1) + 1;
    dim3 grid((unsigned)n_pairs, (unsigned)((pitch / 4 + K5T - 1) / K5T));
    es_perturb_mirrored_kernel<<<grid, K5T, 0, (cudaStream_t)stream>>>(
        theta, in_dim, pitch, sigma, sigma_dev, philox_keys(k0, k1), noise_tag(CEV_KIND_ES_MIRROR, role), gen, row0,
        n_rows, out, noise_out);
    return check_cuda(cudaGetLastError(), "es_perturb_mirrored_kernel");
}

int cev_es_update_mirrored_f32(cev_handle* h, const double* fitness, int in_dim, float sigma, const double* sigma_dev,
                               float lr, int64_t n_total, uint64_t seed, int role, uint32_t gen, int64_t row0,
                               int64_t n_rows, float* delta, cev_stream stream) {
    // an empty shard (n_rows == 0, fitness may be null) still writes its all-zero partial delta
    CEV_REQUIRE(h && (fitness || n_rows == 0) && delta, "es_update_mirrored: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_update_mirrored: in_dim must be 8 or 10");
    CEV_REQUIRE(n_total >= 1 && n_rows >= 0 && (sigma_dev || sigma > 0.f), "es_update_mirrored: bad n/sigma");
    CEV_REQUIRE(row0 >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_update_mirrored: bad row range");
    CEV_REQUIRE(aligned16(delta), "es_update_mirrored: 16B alignment");
    CEV_GUARD(h);
    const int64_t pitch = fc_pitch(in_dim);
    int n_split = (int)((n_rows + 63) / 64);
    if (n_split > 16) n_split = 16;
    if (n_split < 1) n_split = 1;
    int rc = ensure_workspace(h, (size_t)n_split * pitch * sizeof(float));
    if (rc) return rc;
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    float* partial = static_cast<float*>(h->workspace);
    dim3 grid((unsigned)((pitch / 4 + PT - 1) / PT), (unsigned)n_split);
    es_update_mirrored_partial_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(
        fitness, in_dim, pitch, sigma, sigma_dev, philox_keys(k0, k1), noise_tag(CEV_KIND_ES_MIRROR, role), gen, row0,
        n_rows, n_split, partial);
    CEV_CUDA(cudaGetLastError());
    es_update_finish_kernel<<<(unsigned)((pitch + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        partial, n_split, pitch, (double)lr, (double)n_total, sigma, sigma_dev, delta);
    return check_cuda(cudaGetLastError(), "es_update_mirrored kernels");
}

int cev_centered_ranks_f64(cev_handle* h, const double* fitness, int64_t P, int64_t row0, int64_t n_rows,
                           double* out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "centered_ranks: null handle");
    CEV_REQUIRE(P >= 1 && row0 >= 0 && n_rows >= 0 && row0 + n_rows <= P, "centered_ranks: need 0 <= row0, "
                "row0 + n_rows <= P (row0 %lld, n_rows %lld, P %lld)", (long long)row0, (long long)n_rows, (long long)P);
    if (n_rows == 0) return CEV_OK;
    CEV_REQUIRE(fitness && out, "centered_ranks: null pointer");
    CEV_GUARD(h);
    centered_ranks_kernel<<<(unsigned)((n_rows + RK_T - 1) / RK_T), RK_T, 0, (cudaStream_t)stream>>>(
        fitness, P, row0, n_rows, out);
    return check_cuda(cudaGetLastError(), "centered_ranks_kernel");
}

int cev_es_apply_f32(cev_handle* h, float* theta, const float* delta, float* m, float* v, int n_segments,
                     const int* in_dims, int optimizer, double lr, float l2_coeff, int t, cev_stream stream) {
    CEV_REQUIRE(h && theta && delta && in_dims, "es_apply: null pointer");
    CEV_REQUIRE(n_segments >= 1 && n_segments <= CEV_MAX_ROLES, "es_apply: need 1 <= n_segments <= %d", CEV_MAX_ROLES);
    CEV_REQUIRE(optimizer == CEV_ES_SGD || optimizer == CEV_ES_ADAM, "es_apply: optimizer must be CEV_ES_SGD or CEV_ES_ADAM");
    CEV_REQUIRE(optimizer == CEV_ES_SGD || (m && v && t >= 1), "es_apply: Adam needs m, v and t >= 1");
    ApplySegments seg{};
    seg.n = n_segments;
    int64_t off = 0;
    for (int s = 0; s < n_segments; ++s) {
        CEV_REQUIRE(in_dims[s] == IN_ADV || in_dims[s] == IN_GOOD, "es_apply: in_dim must be 8 or 10");
        seg.in_dim[s] = in_dims[s];
        off += fc_pitch(in_dims[s]);
        seg.end[s] = off;
    }
    // Adam's bias-corrected step size in fp64, rounded once to fp32
    const double step = optimizer == CEV_ES_ADAM
        ? lr * sqrt(1.0 - pow(CEV_ADAM_BETA2, (double)t)) / (1.0 - pow(CEV_ADAM_BETA1, (double)t)) : lr;
    CEV_GUARD(h);
    es_apply_kernel<<<(unsigned)((off + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        theta, delta, m, v, seg, optimizer == CEV_ES_ADAM, (float)step, l2_coeff);
    return check_cuda(cudaGetLastError(), "es_apply_kernel");
}

int cev_es_perturb_diag_f32(cev_handle* h, const float* theta, const float* sigma, int in_dim, int mirrored,
                            uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                            float* out, float* noise_out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb_diag: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(theta && sigma && out, "es_perturb_diag: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_perturb_diag: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "es_perturb_diag: bad pitch");
    CEV_REQUIRE(aligned16(theta) && aligned16(sigma) && aligned16(out) && aligned16(noise_out),
                "es_perturb_diag: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb_diag: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    const unsigned ny = (unsigned)((pitch / 4 + K5T - 1) / K5T);
    if (mirrored) {
        const int64_t n_pairs = ((row0 + n_rows - 1) >> 1) - (row0 >> 1) + 1;
        es_perturb_diag_kernel<true><<<dim3((unsigned)n_pairs, ny), K5T, 0, (cudaStream_t)stream>>>(
            theta, sigma, in_dim, pitch, philox_keys(k0, k1), noise_tag(CEV_KIND_ES_MIRROR, role), gen, row0, n_rows,
            out, noise_out);
    } else {
        es_perturb_diag_kernel<false><<<dim3((unsigned)n_rows, ny), K5T, 0, (cudaStream_t)stream>>>(
            theta, sigma, in_dim, pitch, philox_keys(k0, k1), noise_tag(CEV_KIND_ES, role), gen, row0, n_rows, out,
            noise_out);
    }
    return check_cuda(cudaGetLastError(), "es_perturb_diag_kernel");
}

int cev_es_update_diag_f32(cev_handle* h, const double* fitness, int in_dim, int mirrored, int64_t n_total,
                           uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, float* g_mu,
                           float* g_sigma, cev_stream stream) {
    // an empty shard (n_rows == 0, fitness may be null) still writes its all-zero partial sums
    CEV_REQUIRE(h && (fitness || n_rows == 0) && g_mu && g_sigma, "es_update_diag: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_update_diag: in_dim must be 8 or 10");
    CEV_REQUIRE(n_total >= 1 && n_rows >= 0, "es_update_diag: bad n");
    CEV_REQUIRE(row0 >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_update_diag: bad row range");
    CEV_REQUIRE(aligned16(g_mu) && aligned16(g_sigma), "es_update_diag: 16B alignment");
    CEV_GUARD(h);
    const int64_t pitch = fc_pitch(in_dim);
    int n_split = (int)((n_rows + 63) / 64);         // the splits of cev_es_update_f32 / cev_es_update_mirrored_f32
    if (n_split > 16) n_split = 16;
    if (n_split < 1) n_split = 1;
    int rc = ensure_workspace(h, (size_t)2 * n_split * pitch * sizeof(float));
    if (rc) return rc;
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    float* partial = static_cast<float*>(h->workspace);
    dim3 grid((unsigned)((pitch / 4 + PT - 1) / PT), (unsigned)n_split);
    if (mirrored)
        es_update_diag_partial_kernel<true><<<grid, PT, 0, (cudaStream_t)stream>>>(
            fitness, in_dim, pitch, philox_keys(k0, k1), noise_tag(CEV_KIND_ES_MIRROR, role), gen, row0, n_rows,
            n_split, partial);
    else
        es_update_diag_partial_kernel<false><<<grid, PT, 0, (cudaStream_t)stream>>>(
            fitness, in_dim, pitch, philox_keys(k0, k1), noise_tag(CEV_KIND_ES, role), gen, row0, n_rows, n_split,
            partial);
    CEV_CUDA(cudaGetLastError());
    es_update_diag_finish_kernel<<<(unsigned)((pitch + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        partial, n_split, pitch, (double)n_total, g_mu, g_sigma);
    return check_cuda(cudaGetLastError(), "es_update_diag kernels");
}

int cev_es_apply_diag_f32(cev_handle* h, float* theta, float* sigma, const float* g_mu, const float* g_sigma,
                          int n_segments, const int* in_dims, float lr, const double* sigma_lr, float sigma_min,
                          float sigma_max, cev_stream stream) {
    CEV_REQUIRE(h && theta && sigma && g_mu && g_sigma && in_dims && sigma_lr, "es_apply_diag: null pointer");
    CEV_REQUIRE(n_segments >= 1 && n_segments <= CEV_MAX_ROLES, "es_apply_diag: need 1 <= n_segments <= %d",
                CEV_MAX_ROLES);
    CEV_REQUIRE(sigma_min > 0.f && sigma_min <= sigma_max, "es_apply_diag: need 0 < sigma_min <= sigma_max");
    ApplySegments seg{};
    DiagEta eta{};
    seg.n = n_segments;
    int64_t off = 0;
    for (int s = 0; s < n_segments; ++s) {
        CEV_REQUIRE(in_dims[s] == IN_ADV || in_dims[s] == IN_GOOD, "es_apply_diag: in_dim must be 8 or 10");
        CEV_REQUIRE(sigma_lr[s] > 0.0 && std::isfinite(sigma_lr[s]), "es_apply_diag: sigma_lr must be finite and > 0");
        seg.in_dim[s] = in_dims[s];
        eta.half[s] = 0.5 * sigma_lr[s];
        off += fc_pitch(in_dims[s]);
        seg.end[s] = off;
    }
    CEV_GUARD(h);
    es_apply_diag_kernel<<<(unsigned)((off + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        theta, sigma, g_mu, g_sigma, seg, eta, lr, sigma_min, sigma_max);
    return check_cuda(cudaGetLastError(), "es_apply_diag_kernel");
}

int cev_axpy_f32(cev_handle* h, float a, const float* x, float* y, int64_t n, cev_stream stream) {
    CEV_REQUIRE(h && x && y && n >= 0, "axpy: bad arguments");
    if (n == 0) return CEV_OK;
    CEV_GUARD(h);
    axpy_kernel<<<(unsigned)((n + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(a, x, y, n);
    return check_cuda(cudaGetLastError(), "axpy_kernel");
}

int cev_diversity_dist_f32(cev_handle* h, const float* pop, int64_t n_rows, int64_t pitch, const float* ref,
                           int in_dim, float* dist, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "diversity_dist: null handle");
    if (n_rows <= 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(pop && ref && dist, "diversity_dist: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "diversity_dist: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "diversity_dist: bad pitch");
    CEV_REQUIRE(aligned16(pop) && aligned16(ref), "diversity_dist: 16B alignment");
    CEV_GUARD(h);
    diversity_dist_kernel<<<(unsigned)n_rows, PT, 0, (cudaStream_t)stream>>>(pop, pitch, ref, in_dim, dist);
    return check_cuda(cudaGetLastError(), "diversity_dist_kernel");
}

int cev_fc_init_f32(cev_handle* h, int in_dim, uint64_t seed, int role, int64_t row0, int64_t n_rows,
                    int64_t pitch, float* out, cev_stream stream) {
    CEV_REQUIRE(h && out, "fc_init: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "fc_init: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0 && aligned16(out), "fc_init: bad pitch / alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "fc_init: bad row range");
    if (n_rows == 0) return CEV_OK;
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    dim3 grid((unsigned)n_rows, (unsigned)((pitch / 4 + PT - 1) / PT));
    fc_init_kernel<<<grid, PT, 0, (cudaStream_t)stream>>>(in_dim, pitch, k0, k1, noise_tag(4, role), row0, out);
    return check_cuda(cudaGetLastError(), "fc_init_kernel");
}

int cev_init_states_f64(cev_handle* h, uint64_t seed, uint32_t stream_id, int64_t rec0, int64_t n, double* out,
                        cev_stream stream) {
    CEV_REQUIRE(h && (out || n == 0) && n >= 0 && rec0 >= 0 && rec0 + n <= 0xFFFFFFFFll, "init_states: bad arguments");
    if (n == 0) return CEV_OK;
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    init_states_kernel<<<(unsigned)((n + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(k0, k1, stream_id, rec0, n,
                                                                                       out);
    return check_cuda(cudaGetLastError(), "init_states_kernel");
}

int cev_random_frames_u8(cev_handle* h, uint64_t seed, int64_t n_bytes, uint8_t* out, cev_stream stream) {
    CEV_REQUIRE(h && out && n_bytes >= 0 && n_bytes % 16 == 0 && aligned16(out), "random_frames: bad arguments");
    if (n_bytes == 0) return CEV_OK;
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    const int64_t n16 = n_bytes / 16;
    random_frames_kernel<<<(unsigned)((n16 + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        k0, k1, n16, reinterpret_cast<uint4*>(out));
    return check_cuda(cudaGetLastError(), "random_frames_kernel");
}

int cev_philox_words(cev_handle* h, uint64_t seed, int kind, int role, uint32_t gen, int64_t member0,
                     int64_t n_members, int64_t n4, uint32_t* out, cev_stream stream) {
    CEV_REQUIRE(h && out && n_members >= 0 && n4 >= 0 && aligned16(out), "philox_words: bad arguments");
    if (n_members * n4 == 0) return CEV_OK;
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    const int64_t n = n_members * n4;
    philox_words_kernel<<<(unsigned)((n + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        k0, k1, noise_tag(kind, role), gen, member0, n_members, n4, reinterpret_cast<uint4*>(out));
    return check_cuda(cudaGetLastError(), "philox_words_kernel");
}

int cev_es_hof_opponents_i64(cev_handle* h, uint64_t seed, uint32_t gen, int K, int64_t filled, int64_t newest,
                             int64_t* out, cev_stream stream) {
    CEV_REQUIRE(h && out, "es_hof_opponents: null pointer");
    CEV_REQUIRE(K >= 1, "es_hof_opponents: need K >= 1, got %d", K);
    CEV_REQUIRE(filled >= 1 && filled <= 0x100000000ll, "es_hof_opponents: need 1 <= filled <= 2^32, got %lld",
                (long long)filled);
    CEV_REQUIRE(newest >= 0 && newest < filled, "es_hof_opponents: need 0 <= newest < filled");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    es_hof_opponents_kernel<<<(unsigned)((K + PT - 1) / PT), PT, 0, (cudaStream_t)stream>>>(
        k0, k1, gen, K, (uint64_t)filled, newest, out);
    return check_cuda(cudaGetLastError(), "es_hof_opponents_kernel");
}

int cev_weight_stats_f32(cev_handle* h, const float* rows, int64_t n_rows, int64_t pitch, int in_dim, float* out,
                         cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "weight_stats: null handle");
    if (n_rows <= 0) return CEV_OK;
    CEV_REQUIRE(rows && out, "weight_stats: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "weight_stats: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0 && aligned16(rows) && aligned16(out),
                "weight_stats: bad pitch / alignment");
    CEV_GUARD(h);
    weight_stats_kernel<<<(unsigned)n_rows, PT, 0, (cudaStream_t)stream>>>(rows, pitch, in_dim, out);
    return check_cuda(cudaGetLastError(), "weight_stats_kernel");
}

int cev_generation_state_doubles(int hist_capacity) {
    return hist_capacity < 0 ? -1 : CEV_GS_HIST + 3 * hist_capacity + 3 * (hist_capacity + 1);
}

int cev_generation_end_f64(cev_handle* h, const double* eval_out, int n_games, int agent_step_limit,
                           int reference_compat, double* gstate, int hist_capacity, int adaptive, double sigma_max,
                           double sigma_min, int early_stopping, double min_delta, int patience, cev_stream stream) {
    CEV_REQUIRE(h && eval_out && gstate, "generation_end: null pointer");
    CEV_REQUIRE(n_games >= 1 && hist_capacity >= 0, "generation_end: need n_games >= 1, hist_capacity >= 0");
    CEV_GUARD(h);
    generation_end_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(eval_out, n_games, agent_step_limit, reference_compat,
                                                             gstate, hist_capacity, adaptive, sigma_max, sigma_min,
                                                             early_stopping, min_delta, patience);
    return check_cuda(cudaGetLastError(), "generation_end_kernel");
}

int cev_fp32_peak(cev_handle* h, int mode, double* tflops, cev_stream stream) {
    CEV_REQUIRE(h && tflops, "fp32_peak: null pointer");
    CEV_GUARD(h);
    int rc = ensure_workspace(h, 256);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int iters = 4096, blocks = h->n_sm * 8;
    cudaEvent_t e0, e1;
    CEV_CUDA(cudaEventCreate(&e0));
    CEV_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CEV_CUDA(cudaEventRecord(e0, st));
        if (mode == 1) fp32_peak_kernel<1><<<blocks, 256, 0, st>>>((float*)h->workspace, iters);
        else fp32_peak_kernel<0><<<blocks, 256, 0, st>>>((float*)h->workspace, iters);
        CEV_CUDA(cudaEventRecord(e1, st));
        CEV_CUDA(cudaEventSynchronize(e1));
        float ms = 0.f;
        CEV_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flops = (double)blocks * 256.0 * iters * 16.0 * 2.0;
    *tflops = flops / (best * 1e-3) / 1e12;
    return CEV_OK;
}

}  // extern "C"
