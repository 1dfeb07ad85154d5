// Co-ES limited-memory matrix adaptation (LM-MA-ES, Loshchilov, Glasmachers & Beyer 2019): the projection of the
// members' normals on the direction vectors and their transform coefficients (cev_es_lmma_project_f32), the LM-MA K5
// (cev_es_perturb_lmma_f32), the weighted recombination of the selected normals (cev_es_lmma_reduce_f32) and the
// apply with the path, vector, Gram and step-size updates (cev_es_lmma_apply_f32).  A translation unit of its own, so
// every kernel of the other modules keeps its register allocation and SASS.
#include <algorithm>

#include "common.cuh"
#include "es_perturb.cuh"

namespace cev {

constexpr int LM_ROWS = 64;          // members (threads) per projection CTA
constexpr int LM_CHUNK = 2048;       // columns per projection partial sum (fixed: the summation order)
constexpr int LM_SUB = 256;          // columns of M per shared-memory sub-tile of the projection
constexpr int LM_ROWS5 = 32;         // member rows per LM-MA K5 CTA
constexpr int LM_T = 256;            // threads of the reduction, apply and finish kernels
constexpr int LM_SPLIT = 8;          // rank splits of the reduction (fixed: the summation order)
constexpr int LM_ACHUNK = 4096;      // columns per apply CTA (fixed: the summation order of the Gram and |p|^2)
constexpr int LM_ATILE = 256;        // columns per shared-memory tile of the apply
constexpr int LM_MAX = CEV_SUBSPACE_MAX_DIM;

// The step-size constants of the transform: cd[j] = c_d,j and omcd[j] = 1 - c_d,j, computed in fp64 on the host.
struct LmmaDecay {
    double cd[LM_MAX];
    double omcd[LM_MAX];
};

// ---------------------------------------------------------------------------
// 1. Projection: part[c][i][l] = sum over the Linear entries j of column chunk c, in column order from +0, of
//    fma(M[l][j], z_i[j], .) in fp64 (exact fp32 x fp32 products, one rounding per add).  One thread per member: the
//    order does not depend on the CTA, the grid, row0 or n_rows.  M sub-tiles sit in shared memory, read from L2 once
//    per CTA, and are read by every member of the CTA as broadcasts.
// ---------------------------------------------------------------------------
template <int KB>
__global__ void __launch_bounds__(LM_ROWS) lmma_project_kernel(
    const float* __restrict__ M, int64_t ldm, int k, int in_dim, const PhiloxKeys keys, uint32_t tag, uint32_t gen,
    int64_t row0, int64_t n_rows, int n_chunks, double* __restrict__ part) {
    __shared__ float4 sm[KB][LM_SUB / 4];
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r = (int64_t)blockIdx.x * LM_ROWS + threadIdx.x;
    const bool live = r < n_rows;
    const int c = blockIdx.y;
    const int c0 = c * LM_CHUNK, c1 = min(c0 + LM_CHUNK, o.total);
    double acc[KB];
#pragma unroll
    for (int l = 0; l < KB; ++l) acc[l] = 0.0;
    for (int t0 = c0; t0 < c1; t0 += LM_SUB) {
        __syncthreads();
        for (int e = threadIdx.x; e < k * (LM_SUB / 4); e += LM_ROWS) {
            const int l = e / (LM_SUB / 4), q = e - l * (LM_SUB / 4);
            const int j = t0 + 4 * q;
            sm[l][q] = j < c1 ? __ldg(reinterpret_cast<const float4*>(M + l * ldm + j)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        __syncthreads();
        if (!live) continue;
        const int nq = min(LM_SUB, c1 - t0 + 3) / 4;
        for (int q = 0; q < nq; ++q) {
            const int j = t0 + 4 * q;
            if (!fc_is_perturbable(o, j)) continue;
            float z[4];
            normal4(keys, tag, gen, (uint32_t)(row0 + r), (uint32_t)(j >> 2), z);
            const int n_in = min(4, o.total - j);
#pragma unroll
            for (int l = 0; l < KB; ++l) {
                if (l < k) {
                    const float4 mv = sm[l][q];
                    const float m4[4] = {mv.x, mv.y, mv.z, mv.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (i < n_in) acc[l] = fma((double)m4[i], (double)z[i], acc[l]);
                }
            }
        }
    }
    if (!live) return;
    double* out = part + ((int64_t)c * n_rows + r) * k;
#pragma unroll
    for (int l = 0; l < KB; ++l)
        if (l < k) out[l] = acc[l];
}

// s_l = the chunks of the projection summed in order (fp64), then the compact form of the sequential transform:
//   alpha = 1, beta = 0; for j < k: q = alpha s_j + sum_{l < j} beta_l G[j][l] (in order); beta_l *= 1 - c_d,j for
//   l < j; beta_j = c_d,j q; alpha *= 1 - c_d,j
// every operation one IEEE fp64 rounding (no contraction), beta rounded to fp32 once.  A non-finite s or beta sets
// the status word.
__global__ void __launch_bounds__(LM_T) lmma_coef_kernel(const double* __restrict__ part, int n_chunks, int64_t n_rows,
                                                         int k, const double* __restrict__ G, int ldg,
                                                         const LmmaDecay dec, float* __restrict__ beta,
                                                         double* __restrict__ s_out, int* __restrict__ status) {
    const int64_t r = (int64_t)blockIdx.x * LM_T + threadIdx.x;
    if (r >= n_rows) return;
    double s[LM_MAX], b[LM_MAX];
    bool fin = true;
    for (int l = 0; l < k; ++l) {
        double v = 0.0;
        for (int c = 0; c < n_chunks; ++c) v = __dadd_rn(v, part[((int64_t)c * n_rows + r) * k + l]);
        s[l] = v;
        fin = fin && isfinite(v);
        if (s_out) s_out[r * k + l] = v;
    }
    double alpha = 1.0;
    for (int j = 0; j < k; ++j) {
        double q = __dmul_rn(alpha, s[j]);
        for (int l = 0; l < j; ++l) q = __dadd_rn(q, __dmul_rn(b[l], __ldg(G + j * ldg + l)));
        for (int l = 0; l < j; ++l) b[l] = __dmul_rn(b[l], dec.omcd[j]);
        b[j] = __dmul_rn(dec.cd[j], q);
        alpha = __dmul_rn(alpha, dec.omcd[j]);
    }
    for (int l = 0; l < k; ++l) {
        const float f = (float)b[l];
        fin = fin && isfinite(f);
        beta[r * k + l] = f;
    }
    if (!fin && status) atomicOr(status, CEV_STATUS_NONFINITE);
}

// ---------------------------------------------------------------------------
// 2. LM-MA K5: eps = fl(fl(A z) + S), S = sum_{l < k} fl(M[l][j] beta_l) in order from +0 (the guided-search K5's
//    arithmetic with B = 1), member = theta + fl(sigma eps).  A CTA owns a column tile and LM_ROWS5 members and keeps
//    its k float4s of M per thread and the members' beta in shared memory.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(K5T) lmma_perturb_kernel(
    const float* __restrict__ theta, int in_dim, int64_t pitch, const double* __restrict__ sigma_dev,
    const float* __restrict__ M, int64_t ldm, int k, const float* __restrict__ beta, float A, const PhiloxKeys keys,
    uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows, float* __restrict__ out) {
    extern __shared__ float4 lm_smem[];
    float4* su = lm_smem;                                                   // [k][K5T]
    float* sb = reinterpret_cast<float*>(lm_smem + (int64_t)k * K5T);       // [LM_ROWS5][k]
    const float sigma = pick_sigma(0.f, sigma_dev);
    const FcOffsets o = fc_offsets(in_dim);
    const int64_t r0 = (int64_t)blockIdx.x * LM_ROWS5;
    const int n_units = (int)min((int64_t)LM_ROWS5, n_rows - r0);
    const int j4 = blockIdx.y * K5T + threadIdx.x;
    const bool active = (int64_t)j4 * 4 < pitch;
    for (int t = threadIdx.x; t < n_units * k; t += K5T) sb[t] = beta[r0 * k + t];
    if (active)
        for (int l = 0; l < k; ++l) su[l * K5T + threadIdx.x] = __ldg(reinterpret_cast<const float4*>(M + l * ldm) + j4);
    __syncthreads();
    if (!active) return;
    const ScalarSigma sig{sigma};
    for (int u = 0; u < n_units; ++u) {
        const int64_t r = r0 + u;
        SubspaceDir dir{A, 1.f, {0.f, 0.f, 0.f, 0.f}};
        const float* bu = sb + u * k;
        for (int l = 0; l < k; ++l) {
            const float4 mv = su[l * K5T + threadIdx.x];
            const float bl = bu[l];
            dir.s[0] = __fadd_rn(dir.s[0], __fmul_rn(mv.x, bl));
            dir.s[1] = __fadd_rn(dir.s[1], __fmul_rn(mv.y, bl));
            dir.s[2] = __fadd_rn(dir.s[2], __fmul_rn(mv.z, bl));
            dir.s[3] = __fadd_rn(dir.s[3], __fmul_rn(mv.w, bl));
        }
        es_perturb_float4<false>(theta, o, j4, sig, keys, tag, gen, (uint32_t)(row0 + r), out + r * pitch, nullptr,
                                 nullptr, nullptr, dir);
    }
}

// ---------------------------------------------------------------------------
// 3. Weighted recombination of the mu selected members (ids in rank order, weights fp32 w[rank]) over this rank's
//    rows: part[sp][j] = sum over the ranks of split sp, in rank order, of fma(w, z_id[j], .) in fp64 (exact
//    products); members owned by other ranks add nothing.  The finish sums the splits in order and rounds to fp32;
//    block 0 also writes betabar[l] = fp32(sum over the local selected members in rank order of fma(w, beta_id[l], .)).
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(LM_T) lmma_reduce_kernel(const int64_t* __restrict__ ids, const float* __restrict__ w,
                                                           int mu, int in_dim, int64_t pitch, const PhiloxKeys keys,
                                                           uint32_t tag, uint32_t gen, int64_t row0, int64_t n_rows,
                                                           double* __restrict__ part) {
    const int j4 = blockIdx.x * LM_T + threadIdx.x;
    if ((int64_t)j4 * 4 >= pitch) return;
    const int sp = blockIdx.y;
    const int per = (mu + LM_SPLIT - 1) / LM_SPLIT;
    const int a0 = sp * per, a1 = min(mu, a0 + per);
    const FcOffsets o = fc_offsets(in_dim);
    const int j = j4 * 4;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    if (j < o.total && fc_is_perturbable(o, j)) {
        for (int a = a0; a < a1; ++a) {
            const int64_t id = __ldg(ids + a);
            if (id < row0 || id >= row0 + n_rows) continue;
            const double wa = (double)__ldg(w + a);
            float z[4];
            normal4(keys, tag, gen, (uint32_t)id, (uint32_t)j4, z);
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i] = fma(wa, (double)z[i], acc[i]);
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (j + i >= o.total) acc[i] = 0.0;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) part[(int64_t)sp * pitch + j + i] = acc[i];
}

__global__ void __launch_bounds__(LM_T) lmma_reduce_finish_kernel(const double* __restrict__ part, int64_t pitch,
                                                                  const int64_t* __restrict__ ids,
                                                                  const float* __restrict__ w, int mu,
                                                                  const float* __restrict__ beta, int k, int64_t row0,
                                                                  int64_t n_rows, float* __restrict__ zbar,
                                                                  float* __restrict__ betabar) {
    const int64_t j = (int64_t)blockIdx.x * LM_T + threadIdx.x;
    if (j < pitch) {
        double s = 0.0;
        for (int sp = 0; sp < LM_SPLIT; ++sp) s = __dadd_rn(s, part[(int64_t)sp * pitch + j]);
        zbar[j] = (float)s;
    }
    if (blockIdx.x == 0 && threadIdx.x < k) {
        double s = 0.0;
        for (int a = 0; a < mu; ++a) {
            const int64_t id = ids[a];
            if (id < row0 || id >= row0 + n_rows) continue;
            s = fma((double)w[a], (double)beta[(id - row0) * k + threadIdx.x], s);
        }
        betabar[threadIdx.x] = (float)s;
    }
}

// ---------------------------------------------------------------------------
// 4. Apply, per role (segment) of the concatenated rows, on the Linear entries, every operation one IEEE fp64
//    rounding, stores rounded to fp32 once:
//      dbar    = alpha zbar + sum_{l < k} betabar_l M[l]            (in order, M before its update)
//      theta  += (c_m fp32(sigma)) dbar
//      p       = (1 - c_s) p + sqrt(mu_w c_s (2 - c_s)) zbar
//      M[l]    = (1 - c_c,l) M[l] + sqrt(mu_w c_c,l (2 - c_c,l)) zbar     for every l < m
//    and the partial sums over the CTA's column chunk (column order, fp64 products of the new fp32 values) of the new
//    Gram's upper triangle and of |p|^2.  lmma_finish_kernel sums the chunks in order, writes G and adapts sigma.
// ---------------------------------------------------------------------------
struct LmmaRole {
    int in_dim;
    int64_t start, end;          // the segment in the concatenated row
    double alpha, omcs, csq, cm, cs_half, n;
    double omcc[LM_MAX], ccsq[LM_MAX];
};
struct LmmaRoles {
    int n_seg, m, k;
    LmmaRole r[CEV_MAX_ROLES];
};

__global__ void __launch_bounds__(LM_T) lmma_apply_kernel(float* __restrict__ theta, float* __restrict__ M,
                                                          int64_t ldm, float* __restrict__ p,
                                                          const float* __restrict__ zbar,
                                                          const float* __restrict__ betabar,
                                                          const double* __restrict__ gstate, const LmmaRoles roles,
                                                          int n_chunks, double* __restrict__ part) {
    __shared__ float tile[LM_MAX + 1][LM_ATILE + 1];
    const int s = blockIdx.y, m = roles.m, k = roles.k;
    const LmmaRole& R = roles.r[s];
    const FcOffsets o = fc_offsets(R.in_dim);
    const int64_t len = R.end - R.start;
    const int64_t c0 = (int64_t)blockIdx.x * LM_ACHUNK;
    const double step = __dmul_rn(R.cm, (double)(float)gstate[CEV_GS_SIGMA + s]);
    const float* bb = betabar + s * m;
    // this thread's entries (a, b), a <= b < m, of the upper triangle in row-major order, then the entry (m, m): |p|^2
    const int n_pairs = m * (m + 1) / 2 + 1;
    int ea[3], eb[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        int e = threadIdx.x + i * LM_T, a = 0;
        ea[i] = eb[i] = -1;
        if (e >= n_pairs) continue;
        if (e == n_pairs - 1) { ea[i] = eb[i] = m; continue; }
        while (e >= m - a) { e -= m - a; ++a; }
        ea[i] = a;
        eb[i] = a + e;
    }
    double acc[3] = {0.0, 0.0, 0.0};
    for (int64_t t0 = c0; t0 < min(c0 + LM_ACHUNK, len); t0 += LM_ATILE) {
        const int64_t jj = t0 + threadIdx.x;
        const bool pert = jj < len && jj < o.total && fc_is_perturbable(o, (int)jj);
        __syncthreads();
        if (pert) {
            const int64_t i = R.start + jj;
            const double zb = (double)zbar[i];
            double d = __dmul_rn(R.alpha, zb);
            for (int l = 0; l < k; ++l) d = __dadd_rn(d, __dmul_rn((double)bb[l], (double)M[l * ldm + i]));
            theta[i] = (float)__dadd_rn((double)theta[i], __dmul_rn(step, d));
            const float pn = (float)__dadd_rn(__dmul_rn(R.omcs, (double)p[i]), __dmul_rn(R.csq, zb));
            p[i] = pn;
            tile[m][threadIdx.x] = pn;
            for (int l = 0; l < m; ++l) {
                const float v = (float)__dadd_rn(__dmul_rn(R.omcc[l], (double)M[l * ldm + i]), __dmul_rn(R.ccsq[l], zb));
                M[l * ldm + i] = v;
                tile[l][threadIdx.x] = v;
            }
        } else {
            for (int l = 0; l <= m; ++l) tile[l][threadIdx.x] = 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (ea[i] < 0) continue;
            double x = acc[i];
            for (int col = 0; col < LM_ATILE; ++col) x = fma((double)tile[ea[i]][col], (double)tile[eb[i]][col], x);
            acc[i] = x;
        }
    }
    double* out = part + ((int64_t)s * n_chunks + blockIdx.x) * n_pairs;
    const int n_tri = n_pairs - 1;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        if (ea[i] < 0) continue;
        const int e = ea[i] == m ? n_tri : threadIdx.x + i * LM_T;
        out[e] = acc[i];
    }
}

// One CTA per role: G[s][a][b] = G[s][b][a] = the chunks summed in order; |p|^2 likewise; then
//   sigma = clamp(sigma exp(c_s / 2 (|p|^2 / n - 1)), sigma_min, sigma_max)
// into the generation state, stats[s] = (|p|^2 / n, sigma).  A non-finite |p|^2 or Gram entry sets the status word and
// leaves sigma unchanged.
__global__ void __launch_bounds__(LM_T) lmma_finish_kernel(const double* __restrict__ part, int n_chunks,
                                                           const LmmaRoles roles, double* __restrict__ G,
                                                           double* __restrict__ gstate, double sigma_min,
                                                           double sigma_max, double* __restrict__ stats,
                                                           int* __restrict__ status) {
    const int s = blockIdx.x, m = roles.m;
    const int n_pairs = m * (m + 1) / 2 + 1;
    const double* ps = part + (int64_t)s * n_chunks * n_pairs;
    __shared__ int bad;
    if (threadIdx.x == 0) bad = 0;
    __syncthreads();
    for (int e = threadIdx.x; e < n_pairs - 1; e += LM_T) {
        int a = 0, r = e;
        while (r >= m - a) { r -= m - a; ++a; }
        const int b = a + r;
        double v = 0.0;
        for (int c = 0; c < n_chunks; ++c) v = __dadd_rn(v, ps[(int64_t)c * n_pairs + e]);
        if (!isfinite(v)) bad = 1;
        G[((int64_t)s * m + a) * m + b] = v;
        G[((int64_t)s * m + b) * m + a] = v;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double p2 = 0.0;
    for (int c = 0; c < n_chunks; ++c) p2 = __dadd_rn(p2, ps[(int64_t)c * n_pairs + n_pairs - 1]);
    const LmmaRole& R = roles.r[s];
    const double v = p2 / R.n;
    double sigma = gstate[CEV_GS_SIGMA + s];
    if (isfinite(v) && !bad) {
        sigma = sigma * exp(R.cs_half * (v - 1.0));
        sigma = fmin(fmax(sigma, sigma_min), sigma_max);
        gstate[CEV_GS_SIGMA + s] = sigma;
    } else if (status) {
        atomicOr(status, CEV_STATUS_NONFINITE);
    }
    stats[2 * s] = v;
    stats[2 * s + 1] = sigma;
}

}  // namespace cev

using namespace cev;

static bool lm_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static inline PhiloxKeys lm_keys(uint64_t seed) {
    return philox_keys((uint32_t)(seed & 0xFFFFFFFFull), (uint32_t)(seed >> 32));
}

extern "C" {

int cev_es_lmma_project_f32(cev_handle* h, const float* M, int64_t ldm, int k, const double* G, int ldg,
                            const double* cd, int in_dim, uint64_t seed, int role, uint32_t gen, int64_t row0,
                            int64_t n_rows, double* part, float* beta, double* s_out, int* status,
                            cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_lmma_project: null handle");
    if (n_rows == 0) return CEV_OK;
    CEV_REQUIRE(M && G && cd && part && beta, "es_lmma_project: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_lmma_project: in_dim must be 8 or 10");
    CEV_REQUIRE(k >= 1 && k <= CEV_SUBSPACE_MAX_DIM && ldg >= k && ldg <= CEV_SUBSPACE_MAX_DIM,
                "es_lmma_project: need 1 <= k <= ldg <= %d", CEV_SUBSPACE_MAX_DIM);
    CEV_REQUIRE(ldm >= fc_pitch(in_dim) && ldm % 4 == 0 && lm_aligned16(M),
                "es_lmma_project: M needs ldm >= pitch, a multiple of 4, and 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows > 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_lmma_project: bad row range");
    CEV_GUARD(h);
    LmmaDecay dec{};
    for (int j = 0; j < k; ++j) { dec.cd[j] = cd[j]; dec.omcd[j] = 1.0 - cd[j]; }
    const int n_chunks = (fc_offsets(in_dim).total + LM_CHUNK - 1) / LM_CHUNK;
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid((unsigned)((n_rows + LM_ROWS - 1) / LM_ROWS), (unsigned)n_chunks);
    const PhiloxKeys keys = lm_keys(seed);
    const uint32_t tag = noise_tag(CEV_KIND_ES, role);
    if (k <= 8)
        lmma_project_kernel<8><<<grid, LM_ROWS, 0, st>>>(M, ldm, k, in_dim, keys, tag, gen, row0, n_rows, n_chunks, part);
    else if (k <= 16)
        lmma_project_kernel<16><<<grid, LM_ROWS, 0, st>>>(M, ldm, k, in_dim, keys, tag, gen, row0, n_rows, n_chunks, part);
    else
        lmma_project_kernel<32><<<grid, LM_ROWS, 0, st>>>(M, ldm, k, in_dim, keys, tag, gen, row0, n_rows, n_chunks, part);
    CEV_CUDA(cudaGetLastError());
    lmma_coef_kernel<<<(unsigned)((n_rows + LM_T - 1) / LM_T), LM_T, 0, st>>>(part, n_chunks, n_rows, k, G, ldg, dec,
                                                                             beta, s_out, status);
    return check_cuda(cudaGetLastError(), "es_lmma_project kernels");
}

int cev_es_perturb_lmma_f32(cev_handle* h, const float* theta, int in_dim, const double* sigma_dev, const float* M,
                            int64_t ldm, int k, const float* beta, float alpha, uint64_t seed, int role, uint32_t gen,
                            int64_t row0, int64_t n_rows, int64_t pitch, float* out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb_lmma: null handle");
    if (n_rows == 0) return CEV_OK;
    CEV_REQUIRE(theta && sigma_dev && M && beta && out, "es_perturb_lmma: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_perturb_lmma: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "es_perturb_lmma: bad pitch");
    CEV_REQUIRE(k >= 1 && k <= CEV_SUBSPACE_MAX_DIM, "es_perturb_lmma: need 1 <= k <= %d, got %d",
                CEV_SUBSPACE_MAX_DIM, k);
    CEV_REQUIRE(ldm >= pitch && ldm % 4 == 0, "es_perturb_lmma: need ldm >= pitch, a multiple of 4");
    CEV_REQUIRE(lm_aligned16(theta) && lm_aligned16(M) && lm_aligned16(out), "es_perturb_lmma: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows > 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb_lmma: bad row range");
    CEV_GUARD(h);
    const unsigned ny = (unsigned)((pitch / 4 + K5T - 1) / K5T);
    const size_t smem = (size_t)k * K5T * sizeof(float4) + (size_t)LM_ROWS5 * k * sizeof(float);
    CEV_CUDA(cudaFuncSetAttribute(lmma_perturb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lmma_perturb_kernel<<<dim3((unsigned)((n_rows + LM_ROWS5 - 1) / LM_ROWS5), ny), K5T, smem, (cudaStream_t)stream>>>(
        theta, in_dim, pitch, sigma_dev, M, ldm, k, beta, alpha, lm_keys(seed), noise_tag(CEV_KIND_ES, role), gen,
        row0, n_rows, out);
    return check_cuda(cudaGetLastError(), "lmma_perturb_kernel");
}

int cev_es_lmma_reduce_f32(cev_handle* h, const int64_t* ids, const float* w, int mu, const float* beta, int k,
                           int in_dim, uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows,
                           double* part, float* zbar, float* betabar, cev_stream stream) {
    CEV_REQUIRE(h && ids && w && part && zbar, "es_lmma_reduce: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_lmma_reduce: in_dim must be 8 or 10");
    CEV_REQUIRE(mu >= 1 && k >= 0 && k <= CEV_SUBSPACE_MAX_DIM && (k == 0 || (beta && betabar) || n_rows == 0),
                "es_lmma_reduce: need mu >= 1, 0 <= k <= %d and beta / betabar when k > 0", CEV_SUBSPACE_MAX_DIM);
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_lmma_reduce: bad row range");
    CEV_GUARD(h);
    const int64_t pitch = fc_pitch(in_dim);
    cudaStream_t st = (cudaStream_t)stream;
    lmma_reduce_kernel<<<dim3((unsigned)((pitch / 4 + LM_T - 1) / LM_T), LM_SPLIT), LM_T, 0, st>>>(
        ids, w, mu, in_dim, pitch, lm_keys(seed), noise_tag(CEV_KIND_ES, role), gen, row0, n_rows, part);
    CEV_CUDA(cudaGetLastError());
    lmma_reduce_finish_kernel<<<(unsigned)((pitch + LM_T - 1) / LM_T), LM_T, 0, st>>>(
        part, pitch, ids, w, mu, beta, betabar ? k : 0, row0, n_rows, zbar, betabar);
    return check_cuda(cudaGetLastError(), "es_lmma_reduce kernels");
}

int cev_es_lmma_apply_f32(cev_handle* h, float* theta, float* M, int m, int k, float* p, const float* zbar,
                          const float* betabar, int n_segments, const int* in_dims, const double* alpha,
                          const double* c_sigma, const double* mu_w, double c_m, const double* c_c, double* G,
                          double* gstate, double sigma_min, double sigma_max, double* part, double* stats,
                          int* status, cev_stream stream) {
    CEV_REQUIRE(h && theta && M && p && zbar && betabar && in_dims && alpha && c_sigma && mu_w && c_c && G && gstate &&
                    part && stats, "es_lmma_apply: null pointer");
    CEV_REQUIRE(m >= 1 && m <= CEV_SUBSPACE_MAX_DIM && k >= 0 && k <= m, "es_lmma_apply: need 1 <= m <= %d, 0 <= k <= m",
                CEV_SUBSPACE_MAX_DIM);
    CEV_REQUIRE(n_segments >= 1 && n_segments <= CEV_MAX_ROLES, "es_lmma_apply: need 1 <= n_segments <= %d",
                CEV_MAX_ROLES);
    CEV_REQUIRE(sigma_min <= sigma_max, "es_lmma_apply: need sigma_min <= sigma_max");
    LmmaRoles roles{};
    roles.n_seg = n_segments;
    roles.m = m;
    roles.k = k;
    int64_t n = 0, max_len = 0;
    for (int s = 0; s < n_segments; ++s) {
        CEV_REQUIRE(in_dims[s] == IN_ADV || in_dims[s] == IN_GOOD, "es_lmma_apply: in_dim must be 8 or 10");
        LmmaRole& R = roles.r[s];
        R.in_dim = in_dims[s];
        R.start = n;
        n += fc_pitch(in_dims[s]);
        R.end = n;
        max_len = std::max(max_len, (int64_t)fc_pitch(in_dims[s]));
        const double cs = c_sigma[s];
        CEV_REQUIRE(cs > 0.0 && cs < 1.0 && mu_w[s] >= 1.0, "es_lmma_apply: need 0 < c_sigma < 1 and mu_w >= 1");
        const FcOffsets o = fc_offsets(in_dims[s]);
        R.n = (double)(o.total - 2 * (H1 + H2));
        R.alpha = alpha[s];
        R.omcs = 1.0 - cs;
        R.csq = sqrt(mu_w[s] * cs * (2.0 - cs));
        R.cm = c_m;
        R.cs_half = cs / 2.0;
        for (int l = 0; l < m; ++l) {
            const double cc = c_c[s * m + l];
            R.omcc[l] = 1.0 - cc;
            R.ccsq[l] = sqrt(mu_w[s] * cc * (2.0 - cc));
        }
    }
    CEV_GUARD(h);
    const int n_chunks = (int)((max_len + LM_ACHUNK - 1) / LM_ACHUNK);
    cudaStream_t st = (cudaStream_t)stream;
    lmma_apply_kernel<<<dim3((unsigned)n_chunks, (unsigned)n_segments), LM_T, 0, st>>>(theta, M, n, p, zbar, betabar,
                                                                                      gstate, roles, n_chunks, part);
    CEV_CUDA(cudaGetLastError());
    lmma_finish_kernel<<<(unsigned)n_segments, LM_T, 0, st>>>(part, n_chunks, roles, G, gstate, sigma_min, sigma_max,
                                                               stats, status);
    return check_cuda(cudaGetLastError(), "es_lmma_apply kernels");
}

}  // extern "C"
