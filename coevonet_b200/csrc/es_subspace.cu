// Co-ES guided search: the subspace K5 (cev_es_perturb_subspace_f32) and the orthonormal basis of the subspace
// (cev_es_subspace_basis_f32).  A translation unit of its own: ptxas allocates the registers of the kernels of one
// module together, and these kernels in population_ops.cu changed the allocation of generation_end_kernel there.
#include <algorithm>

#include "common.cuh"
#include "es_perturb.cuh"

namespace cev {

// K5 of guided search in the subspace of past update estimates (Guided ES, Maheswaranathan et al. 2019):
//   eps = fl(fl(A z) + fl(B s)),  s = sum_{m < k_eff} fl(U[m][j] c_m) summed in order m = 0, 1, ...
// on the Linear entries, member = theta + fl(sigma eps) (the odd member of a mirrored pair: theta + (-fl(sigma eps))).
// z is the stream of es_perturb_kernel / es_perturb_mirrored_kernel; c_m is normal m of the unit (member, or pair
// under mirroring) in the Philox stream `ctag`.  With B = 0 (k_eff = 0, or alpha = 1) eps = z: the rows of the
// isotropic K5 bit for bit.
//
// The U c term is a [units x k_eff] x [k_eff x d] product: a CTA owns a column tile of K5T float4s and SUB_UNITS
// units.  Each thread keeps its own k_eff float4s of U in shared memory (read from L2 once per CTA, not once per
// member) and the CTA's c values sit in shared memory too.  Dynamic shared memory: k * K5T float4s of U, then
// SUB_UNITS * 4 * ceil(k / 4) floats of c.
constexpr int SUB_ROWS = 32;       // member rows per CTA: 32 members, or 16 mirrored pairs

// B of every possible k_eff, fp32(sqrt((1 - alpha) d / k_eff)) computed in fp64 on the host (b[0] = 0): the kernel
// picks its entry once k_eff is read from the device, without fp64 arithmetic of its own.
struct SubspaceScale {
    float b[CEV_SUBSPACE_MAX_DIM + 1];
};

template <bool MIRROR>
__global__ void __launch_bounds__(K5T) es_perturb_subspace_kernel(
    const float* __restrict__ theta, int in_dim, int64_t pitch, float sigma_arg, const double* __restrict__ sigma_dev,
    const float* __restrict__ U, int64_t ldu, int k, const int* __restrict__ k_eff_dev, float A,
    const SubspaceScale scale, const PhiloxKeys keys, uint32_t tag, uint32_t ctag, uint32_t gen, int64_t row0, int64_t n_rows,
    float* __restrict__ out, float* __restrict__ noise_out, float* __restrict__ coef_out) {
    extern __shared__ float4 sub_smem[];
    float4* su = sub_smem;                                        // [k][K5T]
    constexpr int UNITS = MIRROR ? SUB_ROWS / 2 : SUB_ROWS;
    const int k4 = (k + 3) >> 2;
    float* sc = reinterpret_cast<float*>(sub_smem + (int64_t)k * K5T);     // [UNITS][4 * k4]
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const FcOffsets o = fc_offsets(in_dim);
    const int ke = min(max(__ldg(k_eff_dev), 0), k);
    const float B = scale.b[ke];
    const bool guided = B != 0.f;
    // units of this CTA: members c0 .. c0 + n_units - 1, or pairs q0 .. q0 + n_units - 1
    int64_t u0, n_units;
    if (!MIRROR) {
        u0 = row0 + (int64_t)blockIdx.x * UNITS;
        n_units = min((int64_t)UNITS, row0 + n_rows - u0);
    } else {
        u0 = (row0 >> 1) + (int64_t)blockIdx.x * UNITS;
        n_units = min((int64_t)UNITS, ((row0 + n_rows - 1) >> 1) - u0 + 1);
    }
    const int j4 = blockIdx.y * K5T + threadIdx.x;
    const bool active = (int64_t)j4 * 4 < pitch;
    const bool write_coef = coef_out != nullptr && blockIdx.y == 0;
    if (guided || write_coef) {
        for (int t = threadIdx.x; t < n_units * k4; t += K5T) {
            const int u = t / k4, m4 = t - u * k4;
            float c[4];
            normal4(keys, ctag, gen, (uint32_t)(u0 + u), (uint32_t)m4, c);
#pragma unroll
            for (int i = 0; i < 4; ++i) sc[u * 4 * k4 + m4 * 4 + i] = c[i];
            if (write_coef) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int m = m4 * 4 + i;
                    if (m >= k) break;
                    if (!MIRROR) {
                        coef_out[(u0 + u - row0) * k + m] = c[i];
                    } else {
                        const int64_t rp = 2 * (u0 + u) - row0;
                        if (rp >= 0) coef_out[rp * k + m] = c[i];
                        if (rp + 1 < n_rows) coef_out[(rp + 1) * k + m] = -c[i];
                    }
                }
            }
        }
        if (guided && active)
            for (int m = 0; m < ke; ++m)
                su[m * K5T + threadIdx.x] = __ldg(reinterpret_cast<const float4*>(U + m * ldu) + j4);
        __syncthreads();
    }
    if (!active) return;
    const ScalarSigma sig{sigma};
    for (int u = 0; u < n_units; ++u) {
        const int64_t unit = u0 + u;
        float* plus;
        float* minus = nullptr;
        float* np_ = nullptr;
        float* nm_ = nullptr;
        if (!MIRROR) {
            const int64_t r = unit - row0;
            plus = out + r * pitch;
            if (noise_out) np_ = noise_out + r * pitch;
        } else {
            const int64_t rp = 2 * unit - row0, rm = rp + 1;
            plus = rp >= 0 ? out + rp * pitch : nullptr;
            minus = rm < n_rows ? out + rm * pitch : nullptr;
            if (noise_out && rp >= 0) np_ = noise_out + rp * pitch;
            if (noise_out && rm < n_rows) nm_ = noise_out + rm * pitch;
        }
        if (guided) {
            SubspaceDir dir{A, B, {0.f, 0.f, 0.f, 0.f}};
            const float* cu = sc + u * 4 * k4;
            for (int m = 0; m < ke; ++m) {
                const float4 uv = su[m * K5T + threadIdx.x];
                const float cm = cu[m];
                dir.s[0] = __fadd_rn(dir.s[0], __fmul_rn(uv.x, cm));
                dir.s[1] = __fadd_rn(dir.s[1], __fmul_rn(uv.y, cm));
                dir.s[2] = __fadd_rn(dir.s[2], __fmul_rn(uv.z, cm));
                dir.s[3] = __fadd_rn(dir.s[3], __fmul_rn(uv.w, cm));
            }
            es_perturb_float4<MIRROR>(theta, o, j4, sig, keys, tag, gen, (uint32_t)unit, plus, minus, np_, nm_, dir);
        } else {
            es_perturb_float4<MIRROR>(theta, o, j4, sig, keys, tag, gen, (uint32_t)unit, plus, minus, np_, nm_);
        }
    }
}

// ---------------------------------------------------------------------------
// Orthonormal basis of the guided-search subspace (CholeskyQR2 in fp64 with a column drop rule), per segment
// (role) of the concatenated rows, over its Linear entries only:
//   1. subspace_gram_kernel: partial Gram matrices D^T D of the source rows over fixed column chunks (fp64 products
//      of fp32 values, summed in column order), one CTA per (chunk, segment);
//   2. subspace_chol_kernel: one warp per segment sums the chunks in order and runs a right-looking Cholesky that
//      drops column a when its squared residual is <= 1e-8 of its squared norm (residual norm <= 1e-4 of its own
//      norm; a zero or non-finite column is always dropped), then inverts R on the kept columns: T = R^-1;
//   3. subspace_apply_kernel: U = D T, rounded to fp32 once (zero rows past the kept count, zero on LayerNorm
//      entries and padding).
// The chain runs twice: on the ring (rows newest first), then in place on U.
// ---------------------------------------------------------------------------
constexpr int SB_T = 256;          // threads of the Gram and apply kernels
constexpr int SB_TILE = 128;       // columns per shared-memory tile of the Gram kernel
constexpr int SB_CHUNK = 4096;     // columns per Gram CTA
constexpr int SB_KMAX = 32;

// Row a of the source matrix: slot (newest - a) mod k of a ring holding `filled` rows (ring = 1), or row a (ring = 0);
// -1 = a zero row.
struct SubRows {
    int k, newest, filled, ring;
    __device__ __forceinline__ int slot(int a) const {
        if (a >= filled) return -1;
        return ring ? (newest - a + k) % k : a;
    }
};

// Segments (roles) of the concatenated rows: the layout of cev_es_apply_f32.
struct ApplySegments {
    int n;
    int in_dim[CEV_MAX_ROLES];
    int64_t end[CEV_MAX_ROLES];        // exclusive end offset of each segment in the concatenated row
};

__device__ __forceinline__ void segment_of(const ApplySegments& seg, int64_t i, int& s, int& in_dim, int64_t& start,
                                           int64_t& end) {
    s = 0;
    in_dim = seg.in_dim[0];
    start = 0;
    end = seg.end[0];
#pragma unroll
    for (int t = 1; t < CEV_MAX_ROLES; ++t)
        if (t < seg.n && i >= end) { s = t; in_dim = seg.in_dim[t]; start = end; end = seg.end[t]; }
}

__global__ void __launch_bounds__(SB_T) subspace_gram_kernel(const float* __restrict__ src, int64_t ld,
                                                             const SubRows rows, const ApplySegments seg,
                                                             int n_chunks, double* __restrict__ partial) {
    __shared__ float tile[SB_KMAX][SB_TILE + 1];
    const int s = blockIdx.y, k = rows.k;
    const int64_t start = s ? seg.end[s - 1] : 0, len = seg.end[s] - start;
    const FcOffsets o = fc_offsets(seg.in_dim[s]);
    const int64_t c0 = (int64_t)blockIdx.x * SB_CHUNK;
    // this thread's entries (a, b), a <= b, of the upper triangle in row-major order
    int ea[3], eb[3];
    const int n_pairs = k * (k + 1) / 2;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        int e = threadIdx.x + i * SB_T, a = 0;
        ea[i] = eb[i] = -1;
        if (e >= n_pairs) continue;
        while (e >= k - a) { e -= k - a; ++a; }
        ea[i] = a;
        eb[i] = a + e;
    }
    double acc[3] = {0.0, 0.0, 0.0};
    for (int64_t t0 = c0; t0 < min(c0 + SB_CHUNK, len); t0 += SB_TILE) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < k * SB_TILE; idx += SB_T) {
            const int a = idx / SB_TILE, col = idx - a * SB_TILE;
            const int64_t j = t0 + col;
            const int sl = rows.slot(a);
            float v = 0.f;
            if (sl >= 0 && j < len && j < o.total && fc_is_perturbable(o, (int)j)) v = src[sl * ld + start + j];
            tile[a][col] = v;
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            if (ea[i] < 0) continue;
            double x = acc[i];
            for (int col = 0; col < SB_TILE; ++col)
                x = fma((double)tile[ea[i]][col], (double)tile[eb[i]][col], x);
            acc[i] = x;
        }
    }
    double* out = partial + ((int64_t)s * n_chunks + blockIdx.x) * k * k;
#pragma unroll
    for (int i = 0; i < 3; ++i)
        if (ea[i] >= 0) out[ea[i] * k + eb[i]] = acc[i];
}

// One warp per segment.  T (out): fp64 [k][k], T[a][r] = (R^-1)[pos(a)][r] for kept source row a at position pos(a)
// among the kept rows, 0 elsewhere; n_kept (out): the kept count.
__global__ void __launch_bounds__(32) subspace_chol_kernel(const double* __restrict__ partial, int n_chunks, int k,
                                                           double* __restrict__ T, int* __restrict__ n_kept) {
    __shared__ double G[SB_KMAX][SB_KMAX + 1], W[SB_KMAX][SB_KMAX + 1], R[SB_KMAX][SB_KMAX + 1];
    __shared__ int kept[SB_KMAX];
    const int s = blockIdx.x, lane = threadIdx.x;
    const double* p = partial + (int64_t)s * n_chunks * k * k;
    for (int e = lane; e < k * k; e += 32) {
        const int a = e / k, b = e - a * k;
        if (a > b) continue;
        double sum = 0.0;
        for (int c = 0; c < n_chunks; ++c) sum += p[(int64_t)c * k * k + e];
        G[a][b] = G[b][a] = sum;
        W[a][b] = W[b][a] = sum;
        R[a][b] = R[b][a] = 0.0;
    }
    __syncwarp();
    int nk = 0;
    for (int a = 0; a < k; ++a) {
        const double diag = W[a][a];
        if (!(diag > 1e-8 * G[a][a])) continue;          // dependent (or zero / non-finite) estimate: dropped
        const double r = sqrt(diag);
        if (lane >= a && lane < k) R[a][lane] = lane == a ? r : W[a][lane] / r;
        __syncwarp();
        if (lane > a && lane < k)
            for (int c = a + 1; c < k; ++c) W[lane][c] -= R[a][lane] * R[a][c];
        if (lane == 0) kept[nk] = a;
        ++nk;
        __syncwarp();
    }
    // inverse of the kept block Rk[p][q] = R[kept[p]][kept[q]] (upper triangular): lane q solves Rk x = e_q
    double x[SB_KMAX];
#pragma unroll
    for (int i = 0; i < SB_KMAX; ++i) x[i] = 0.0;
    if (lane < nk) {
#pragma unroll
        for (int pp = SB_KMAX - 1; pp >= 0; --pp) {
            if (pp > lane) continue;
            double acc = pp == lane ? 1.0 : 0.0;
#pragma unroll
            for (int t = pp + 1; t < SB_KMAX; ++t)
                if (t <= lane) acc -= R[kept[pp]][kept[t]] * x[t];
            x[pp] = acc / R[kept[pp]][kept[pp]];
        }
    }
    double* Ts = T + (int64_t)s * k * k;
    for (int e = lane; e < k * k; e += 32) Ts[e] = 0.0;
    __syncwarp();
#pragma unroll
    for (int pp = 0; pp < SB_KMAX; ++pp)
        if (pp < nk && lane < nk) Ts[kept[pp] * k + lane] = x[pp];
    if (lane == 0) n_kept[s] = nk;
}

// dst[r][i] = fp32(sum_a T[s][a][r] src_a[i]) for r < n_kept[s], 0 for r >= n_kept[s] and off the Linear entries.
// Terms with T[s][a][r] = 0 are skipped: a dropped source row (T = 0 in every column) never enters U, even when it
// holds an inf or a NaN, and for finite values skipping fma(0, x, v) changes no bit (v starts at +0).
// All k source values of column i are read before any write: src may be dst.
__global__ void __launch_bounds__(SB_T) subspace_apply_kernel(const float* src, int64_t ld, const SubRows rows,
                                                              const ApplySegments seg, const double* __restrict__ T,
                                                              const int* __restrict__ n_kept, float* dst) {
    const int64_t i = (int64_t)blockIdx.x * SB_T + threadIdx.x;
    int s, in_dim;
    int64_t start, end;
    segment_of(seg, i, s, in_dim, start, end);
    if (i >= end) return;
    const int k = rows.k;
    const FcOffsets o = fc_offsets(in_dim);
    const int j = (int)(i - start);
    const bool pert = j < o.total && fc_is_perturbable(o, j);
    const int nk = n_kept[s];
    float x[SB_KMAX];
#pragma unroll
    for (int a = 0; a < SB_KMAX; ++a) {
        const int sl = a < k ? rows.slot(a) : -1;
        x[a] = (pert && sl >= 0) ? src[sl * ld + i] : 0.f;
    }
    const double* Ts = T + (int64_t)s * k * k;
    for (int r = 0; r < k; ++r) {
        double v = 0.0;
        if (pert && r < nk) {
#pragma unroll
            for (int a = 0; a < SB_KMAX; ++a)
                if (a < k) {
                    const double t = __ldg(Ts + a * k + r);
                    if (t != 0.0) v = fma(t, (double)x[a], v);
                }
        }
        dst[r * ld + i] = (float)v;
    }
}

}  // namespace cev

using namespace cev;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static inline void split_seed(uint64_t seed, uint32_t& k0, uint32_t& k1) {
    k0 = (uint32_t)(seed & 0xFFFFFFFFull);
    k1 = (uint32_t)(seed >> 32);
}

extern "C" {

int cev_es_perturb_subspace_f32(cev_handle* h, const float* theta, int in_dim, float sigma, const double* sigma_dev,
                                const float* U, int64_t ldu, int k, const int* k_eff, double alpha, int mirrored,
                                uint64_t seed, int role, uint32_t gen, int64_t row0, int64_t n_rows, int64_t pitch,
                                float* out, float* noise_out, float* coef_out, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "es_perturb_subspace: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(theta && U && k_eff && out, "es_perturb_subspace: null pointer");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "es_perturb_subspace: in_dim must be 8 or 10");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "es_perturb_subspace: bad pitch");
    CEV_REQUIRE(k >= 1 && k <= CEV_SUBSPACE_MAX_DIM, "es_perturb_subspace: need 1 <= k <= %d, got %d",
                CEV_SUBSPACE_MAX_DIM, k);
    CEV_REQUIRE(ldu >= pitch && ldu % 4 == 0, "es_perturb_subspace: need ldu >= pitch, a multiple of 4");
    CEV_REQUIRE(alpha > 0.0 && alpha <= 1.0, "es_perturb_subspace: alpha must be in (0, 1]");
    CEV_REQUIRE(aligned16(theta) && aligned16(U) && aligned16(out) && aligned16(noise_out),
                "es_perturb_subspace: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "es_perturb_subspace: bad row range");
    CEV_GUARD(h);
    uint32_t k0, k1;
    split_seed(seed, k0, k1);
    const float A = (float)sqrt(alpha);
    SubspaceScale scale;
    const double d = (double)(fc_offsets(in_dim).total - 2 * (H1 + H2));       // perturbable entries of the row
    scale.b[0] = 0.f;
    for (int m = 1; m <= CEV_SUBSPACE_MAX_DIM; ++m) scale.b[m] = (float)sqrt((1.0 - alpha) * d / (double)m);
    const unsigned ny = (unsigned)((pitch / 4 + K5T - 1) / K5T);
    const size_t smem = (size_t)k * K5T * sizeof(float4) + (size_t)SUB_ROWS * 4 * ((k + 3) / 4) * sizeof(float);
    cudaStream_t st = (cudaStream_t)stream;
    if (mirrored) {
        const int64_t n_pairs = ((row0 + n_rows - 1) >> 1) - (row0 >> 1) + 1;
        CEV_CUDA(cudaFuncSetAttribute(es_perturb_subspace_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
        es_perturb_subspace_kernel<true><<<dim3((unsigned)((n_pairs + SUB_ROWS / 2 - 1) / (SUB_ROWS / 2)), ny), K5T,
                                           smem, st>>>(
            theta, in_dim, pitch, sigma, sigma_dev, U, ldu, k, k_eff, A, scale, philox_keys(k0, k1),
            noise_tag(CEV_KIND_ES_MIRROR, role), noise_tag(CEV_KIND_ES_SUBSPACE, role), gen, row0, n_rows, out,
            noise_out, coef_out);
    } else {
        CEV_CUDA(cudaFuncSetAttribute(es_perturb_subspace_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
        es_perturb_subspace_kernel<false><<<dim3((unsigned)((n_rows + SUB_ROWS - 1) / SUB_ROWS), ny), K5T, smem,
                                            st>>>(
            theta, in_dim, pitch, sigma, sigma_dev, U, ldu, k, k_eff, A, scale, philox_keys(k0, k1),
            noise_tag(CEV_KIND_ES, role), noise_tag(CEV_KIND_ES_SUBSPACE, role), gen, row0, n_rows, out, noise_out,
            coef_out);
    }
    return check_cuda(cudaGetLastError(), "es_perturb_subspace_kernel");
}

int cev_es_subspace_basis_f32(cev_handle* h, const float* ring, int k, int newest, int filled, int n_segments,
                              const int* in_dims, float* U, int* k_eff, cev_stream stream) {
    CEV_REQUIRE(h && ring && in_dims && U && k_eff, "es_subspace_basis: null pointer");
    CEV_REQUIRE(ring != U, "es_subspace_basis: ring and U must be distinct buffers");
    CEV_REQUIRE(k >= 1 && k <= CEV_SUBSPACE_MAX_DIM, "es_subspace_basis: need 1 <= k <= %d, got %d",
                CEV_SUBSPACE_MAX_DIM, k);
    CEV_REQUIRE(filled >= 0 && filled <= k && newest >= 0 && newest < k,
                "es_subspace_basis: need 0 <= filled <= k and 0 <= newest < k");
    CEV_REQUIRE(n_segments >= 1 && n_segments <= CEV_MAX_ROLES, "es_subspace_basis: need 1 <= n_segments <= %d",
                CEV_MAX_ROLES);
    ApplySegments seg{};
    seg.n = n_segments;
    int64_t n = 0, max_len = 0;
    for (int s = 0; s < n_segments; ++s) {
        CEV_REQUIRE(in_dims[s] == IN_ADV || in_dims[s] == IN_GOOD, "es_subspace_basis: in_dim must be 8 or 10");
        seg.in_dim[s] = in_dims[s];
        n += fc_pitch(in_dims[s]);
        max_len = std::max(max_len, (int64_t)fc_pitch(in_dims[s]));
        seg.end[s] = n;
    }
    CEV_GUARD(h);
    const int n_chunks = (int)((max_len + SB_CHUNK - 1) / SB_CHUNK);
    const size_t kk = (size_t)k * k;
    const size_t part_d = (size_t)n_segments * n_chunks * kk, t_d = (size_t)n_segments * kk;
    const size_t need = (part_d + t_d) * sizeof(double) + CEV_MAX_ROLES * sizeof(int);
    if (h->workspace_bytes < need) {
        if (h->workspace) cudaFree(h->workspace);
        h->workspace = nullptr;
        h->workspace_bytes = 0;
        CEV_CUDA(cudaMalloc(&h->workspace, need));
        h->workspace_bytes = need;
    }
    double* partial = static_cast<double*>(h->workspace);
    double* T = partial + part_d;
    int* kept1 = reinterpret_cast<int*>(T + t_d);
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned n_blocks = (unsigned)((n + SB_T - 1) / SB_T);
    // pass 1: the ring, newest estimate first
    const SubRows from_ring{k, newest, filled, 1};
    subspace_gram_kernel<<<dim3((unsigned)n_chunks, (unsigned)n_segments), SB_T, 0, st>>>(ring, n, from_ring, seg,
                                                                                          n_chunks, partial);
    subspace_chol_kernel<<<(unsigned)n_segments, 32, 0, st>>>(partial, n_chunks, k, T, kept1);
    subspace_apply_kernel<<<n_blocks, SB_T, 0, st>>>(ring, n, from_ring, seg, T, kept1, U);
    CEV_CUDA(cudaGetLastError());
    // pass 2: the same on U, in place
    const SubRows from_u{k, 0, k, 0};
    subspace_gram_kernel<<<dim3((unsigned)n_chunks, (unsigned)n_segments), SB_T, 0, st>>>(U, n, from_u, seg,
                                                                                          n_chunks, partial);
    subspace_chol_kernel<<<(unsigned)n_segments, 32, 0, st>>>(partial, n_chunks, k, T, k_eff);
    subspace_apply_kernel<<<n_blocks, SB_T, 0, st>>>(U, n, from_u, seg, T, k_eff, U);
    return check_cuda(cudaGetLastError(), "es_subspace_basis kernels");
}

}  // extern "C"
