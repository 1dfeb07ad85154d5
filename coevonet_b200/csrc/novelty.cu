// Co-ES novelty search (NS-ES / NSR-ES, Conti et al. 2018) on a policy-space behaviour characterisation: the probe
// observations (cev_novelty_probe_obs_f32), the behaviour characterisation of member rows (cev_novelty_bc_f32) and
// the k-nearest-neighbour novelty against an archive (cev_novelty_knn_f64).  A translation unit of its own: ptxas
// allocates the registers of the kernels of one module together, so apart from them every existing kernel keeps its
// SASS.
#include <algorithm>
#include <climits>

#include "common.cuh"

namespace cev {

constexpr int NV_P = CEV_NOVELTY_PROBES;      // probe observations per behaviour characterisation
constexpr int NV_BC = CEV_NOVELTY_BC_DIM;     // NV_P * NACT floats
constexpr int NV_T = 256;                     // threads of the BC kernel
constexpr int NV_KT = 32;                     // fc2 columns per shared-memory tile of W2
constexpr int NV_OBS_LD = 16;                 // row stride of the probe observations in shared memory
static_assert(NV_BC == NV_P * NACT, "BC layout");
static_assert(NV_T == H2 && 2 * NV_T == H1, "the BC kernel maps threads to units");

// ---------------------------------------------------------------------------------------------------------------
// probe observations: obs[i] = env_observe(env_load(init[i]), seat), the rollout's own observation code
// ---------------------------------------------------------------------------------------------------------------
__global__ void novelty_probe_obs_kernel(const double* __restrict__ init, int64_t n, int seat, float* __restrict__ obs) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    EnvState s;
    env_load(s, init + i * CEV_INIT_STATE_DIM);
    float o[IN_GOOD];
    env_observe(s, seat, o);
    const int in_dim = seat_in_dim(seat);
#pragma unroll
    for (int t = 0; t < IN_GOOD; ++t)
        if (t < in_dim) obs[i * in_dim + t] = o[t];
}

// ---------------------------------------------------------------------------------------------------------------
// BC kernel: one member per CTA job (CTAs loop over members), the 32 probes as the batch.  Every member row is read
// from global memory once: fc1 and the LayerNorm / output vectors by the threads that use them, fc2 (the bulk of the
// row) as coalesced 32-column tiles staged through shared memory, with the next tile in registers while the current
// one is multiplied.  FP32 FFMA throughout.
//
// Shared memory: a1 [32 probes][512] (layer-1 activations), wt [32 k][256 units] (the W2 tile; later the layer-2
// activations [32 probes][256]), the probe observations [32][16].
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// In-place LayerNorm (biased variance, eps 1e-5) + ReLU of the rows p = warp, warp + 8, ... of x [32][N].  A non-finite
// activation stays non-finite, so it reaches the logits and the status word.
template <int N>
__device__ __forceinline__ void layer_norm_relu_rows(float* x, const float* __restrict__ g, const float* __restrict__ b,
                                                     int warp, int lane) {
    constexpr int V = N / 32;
    float gv[V], bv[V];
#pragma unroll
    for (int i = 0; i < V; ++i) {
        gv[i] = __ldg(g + lane + 32 * i);
        bv[i] = __ldg(b + lane + 32 * i);
    }
    for (int p = warp; p < NV_P; p += NV_T / 32) {
        float* row = x + p * N;
        float v[V];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i] = row[lane + 32 * i];
            s += v[i];
        }
        const float mean = warp_sum(s) * (1.0f / N);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < V; ++i) {
            v[i] -= mean;
            q = fmaf(v[i], v[i], q);
        }
        const float var = warp_sum(q) * (1.0f / N);
        const float rstd = 1.0f / sqrtf(var + LN_EPS);
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float y = fmaf(v[i] * rstd, gv[i], bv[i]);
            row[lane + 32 * i] = y < 0.f ? 0.f : y;         // ReLU that keeps a NaN (fmaxf would drop it)
        }
    }
}

template <int IN>
__global__ void __launch_bounds__(NV_T) novelty_bc_kernel(const float* __restrict__ rows, int64_t pitch, int64_t P,
                                                         const float* __restrict__ probe_obs, float* __restrict__ bc,
                                                         int64_t bc_pitch, int32_t* __restrict__ status) {
    extern __shared__ float4 nv_smem[];
    float* a1 = reinterpret_cast<float*>(nv_smem);        // [NV_P][H1]
    float* wt = a1 + NV_P * H1;                           // [NV_KT][H2], then h2 [NV_P][H2]
    float* so = wt + NV_KT * H2;                          // [NV_P][NV_OBS_LD]
    constexpr FcOffsets o = fc_offsets(IN);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < NV_P * IN; i += NV_T) so[(i / IN) * NV_OBS_LD + i % IN] = probe_obs[i];
    // layer-2 thread tile: units j0 .. j0 + 3, probes p0 .. p0 + 7 (a warp shares its probes: broadcast reads of a1)
    const int j0 = 4 * ((warp & 1) * 32 + lane), p0 = 8 * (warp >> 1);
    for (int64_t m = blockIdx.x; m < P; m += gridDim.x) {
        const float* W = rows + m * pitch;
        __syncthreads();                                  // the previous member's readers of a1 / wt are done
        // ---- layer 1: thread owns units tid and tid + 256 ----------------------------------------------------
#pragma unroll
        for (int uu = 0; uu < 2; ++uu) {
            const int u = tid + uu * NV_T;
            float w[IN];
#pragma unroll
            for (int i = 0; i < IN; ++i) w[i] = __ldg(W + o.fc1w + u * IN + i);
            const float b = __ldg(W + o.fc1b + u);
            for (int p = 0; p < NV_P; ++p) {
                float acc = 0.f;
#pragma unroll
                for (int i = 0; i < IN; ++i) acc = fmaf(so[p * NV_OBS_LD + i], w[i], acc);
                a1[p * H1 + u] = acc + b;
            }
        }
        __syncthreads();
        layer_norm_relu_rows<H1>(a1, W + o.ln1g, W + o.ln1b, warp, lane);
        // ---- layer 2: [32 x 512] x [512 x 256]; thread tid stages row tid of W2 ----------------------------------
        const float4* w2row = reinterpret_cast<const float4*>(W + o.fc2w + (int64_t)tid * H1);
        float4 pf[NV_KT / 4];
#pragma unroll
        for (int q = 0; q < NV_KT / 4; ++q) pf[q] = __ldg(w2row + q);
        float acc[8][4];
#pragma unroll
        for (int pp = 0; pp < 8; ++pp)
#pragma unroll
            for (int u = 0; u < 4; ++u) acc[pp][u] = 0.f;
        for (int k0 = 0; k0 < H1; k0 += NV_KT) {
            __syncthreads();                              // LayerNorm 1 written / the previous tile consumed
#pragma unroll
            for (int q = 0; q < NV_KT / 4; ++q) {
                wt[(4 * q + 0) * H2 + tid] = pf[q].x;
                wt[(4 * q + 1) * H2 + tid] = pf[q].y;
                wt[(4 * q + 2) * H2 + tid] = pf[q].z;
                wt[(4 * q + 3) * H2 + tid] = pf[q].w;
            }
            __syncthreads();
            if (k0 + NV_KT < H1) {
#pragma unroll
                for (int q = 0; q < NV_KT / 4; ++q) pf[q] = __ldg(w2row + (k0 + NV_KT) / 4 + q);
            }
#pragma unroll
            for (int kk = 0; kk < NV_KT; kk += 4) {
                float4 wv[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) wv[t] = *reinterpret_cast<const float4*>(wt + (kk + t) * H2 + j0);
#pragma unroll
                for (int pp = 0; pp < 8; ++pp) {
                    const float4 av = *reinterpret_cast<const float4*>(a1 + (p0 + pp) * H1 + k0 + kk);
                    const float a[4] = {av.x, av.y, av.z, av.w};
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        acc[pp][0] = fmaf(a[t], wv[t].x, acc[pp][0]);
                        acc[pp][1] = fmaf(a[t], wv[t].y, acc[pp][1]);
                        acc[pp][2] = fmaf(a[t], wv[t].z, acc[pp][2]);
                        acc[pp][3] = fmaf(a[t], wv[t].w, acc[pp][3]);
                    }
                }
            }
        }
        const float4 b2 = __ldg(reinterpret_cast<const float4*>(W + o.fc2b) + j0 / 4);
        __syncthreads();                                  // every reader of the last W2 tile is done
        float* h2 = wt;
#pragma unroll
        for (int pp = 0; pp < 8; ++pp)
            *reinterpret_cast<float4*>(h2 + (p0 + pp) * H2 + j0) =
                make_float4(acc[pp][0] + b2.x, acc[pp][1] + b2.y, acc[pp][2] + b2.z, acc[pp][3] + b2.w);
        __syncthreads();
        layer_norm_relu_rows<H2>(h2, W + o.ln2g, W + o.ln2b, warp, lane);
        __syncwarp();
        // ---- output layer + softmax: warp per probe (the probes its LayerNorm wrote) ------------------------------
        for (int p = warp; p < NV_P; p += NV_T / 32) {
            float x[H2 / 32];
#pragma unroll
            for (int i = 0; i < H2 / 32; ++i) x[i] = h2[p * H2 + lane + 32 * i];
            float lg[NACT];
#pragma unroll
            for (int a = 0; a < NACT; ++a) {
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < H2 / 32; ++i) s = fmaf(x[i], __ldg(W + o.outw + a * H2 + lane + 32 * i), s);
                lg[a] = warp_sum(s) + __ldg(W + o.outb + a);
            }
            if (lane < NACT) {
                bool fin = true;
                float mx = lg[0];
#pragma unroll
                for (int a = 0; a < NACT; ++a) {
                    fin = fin && isfinite(lg[a]);
                    mx = fmaxf(mx, lg[a]);
                }
                float e[NACT], sum = 0.f;
#pragma unroll
                for (int a = 0; a < NACT; ++a) {
                    e[a] = expf(lg[a] - mx);
                    sum += e[a];
                }
                float mine = e[0];
#pragma unroll
                for (int a = 1; a < NACT; ++a)
                    if (lane == a) mine = e[a];
                bc[m * bc_pitch + p * NACT + lane] = mine / sum;
                if (!fin && lane == 0 && status) atomicOr(status, CEV_STATUS_NONFINITE);
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// k-NN novelty: one warp per member, the archive streamed through shared memory in tiles of 32 entries (lane e of
// the warp measures entry e of the tile), the k smallest (distance, slot) pairs kept sorted across the lanes.
// ---------------------------------------------------------------------------------------------------------------
constexpr int KN_WARPS = 8;
constexpr int KN_TILE = 32;
constexpr int KN_LD = NV_BC + 1;              // padded entry stride: lane e reads bank (e + t) mod 32

__device__ __forceinline__ bool pair_less(double d0, int s0, double d1, int s1) {
    return d0 < d1 || (d0 == d1 && s0 < s1);
}

__global__ void __launch_bounds__(KN_WARPS * 32) novelty_knn_kernel(const float* __restrict__ bc, int64_t n,
                                                                    const float* __restrict__ ring, int filled, int k,
                                                                    double* __restrict__ novelty) {
    __shared__ float sr[KN_TILE * KN_LD];
    __shared__ double sx[KN_WARPS][NV_BC];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * KN_WARPS + warp;
    const bool active = i < n;                                   // warp-uniform
    if (active)
        for (int t = lane; t < NV_BC; t += 32) sx[warp][t] = (double)bc[i * NV_BC + t];
    double ld = CUDART_INF;                                      // lane l: the l-th smallest pair so far
    int ls = INT_MAX;
    for (int e0 = 0; e0 < filled; e0 += KN_TILE) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < KN_TILE * NV_BC; idx += KN_WARPS * 32) {
            const int e = idx / NV_BC, t = idx - e * NV_BC;
            sr[e * KN_LD + t] = e0 + e < filled ? ring[(int64_t)(e0 + e) * NV_BC + t] : 0.f;
        }
        __syncthreads();
        if (!active) continue;
        const int e = e0 + lane;
        const bool valid = e < filled;
        double s = 0.0;
        const float* y = sr + lane * KN_LD;
        for (int t = 0; t < NV_BC; ++t) {
            const double d = __dsub_rn(sx[warp][t], (double)y[t]);
            s = __dadd_rn(s, __dmul_rn(d, d));
        }
        const double dist = __dsqrt_rn(s);
        const double kd = __shfl_sync(0xffffffffu, ld, k - 1);
        const int ks = __shfl_sync(0xffffffffu, ls, k - 1);
        unsigned cand = __ballot_sync(0xffffffffu, valid && pair_less(dist, e, kd, ks));
        while (cand) {
            const int src = __ffs(cand) - 1;
            cand &= cand - 1;
            const double cd = __shfl_sync(0xffffffffu, dist, src);
            const int cs = e0 + src;
            if (!pair_less(cd, cs, __shfl_sync(0xffffffffu, ld, k - 1), __shfl_sync(0xffffffffu, ls, k - 1)))
                continue;                                         // no longer among the k smallest
            const unsigned after = __ballot_sync(0xffffffffu, pair_less(cd, cs, ld, ls));
            const int pos = __ffs(after) - 1;                     // <= k - 1: the candidate beats lane k - 1
            const double up_d = __shfl_up_sync(0xffffffffu, ld, 1);
            const int up_s = __shfl_up_sync(0xffffffffu, ls, 1);
            if (lane > pos) {
                ld = up_d;
                ls = up_s;
            } else if (lane == pos) {
                ld = cd;
                ls = cs;
            }
        }
    }
    if (!active) return;
    const int ke = min(k, filled);
    double sum = 0.0;
    for (int j = 0; j < ke; ++j) sum = __dadd_rn(sum, __shfl_sync(0xffffffffu, ld, j));
    if (lane == 0) novelty[i] = __ddiv_rn(sum, (double)ke);
}

}  // namespace cev

using namespace cev;

static bool nv_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int IN>
static int launch_novelty_bc(cev_handle* h, const float* rows, int64_t pitch, int64_t P, const float* probe_obs,
                             float* bc, int64_t bc_pitch, int32_t* status, cudaStream_t st) {
    const size_t smem = (size_t)(NV_P * H1 + NV_KT * H2 + NV_P * NV_OBS_LD) * sizeof(float);
    // the shared-memory attribute and the resident CTAs per SM, once per device (a function attribute is per device)
    static int per_sm[16] = {};
    int resident = h->device < 16 ? per_sm[h->device] : 0;
    if (resident == 0) {
        CEV_CUDA(cudaFuncSetAttribute(novelty_bc_kernel<IN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        CEV_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, novelty_bc_kernel<IN>, NV_T, smem));
        resident = std::max(resident, 1);
        if (h->device < 16) per_sm[h->device] = resident;
    }
    const int64_t grid = std::min<int64_t>(P, (int64_t)resident * h->n_sm);
    novelty_bc_kernel<IN><<<(unsigned)grid, NV_T, smem, st>>>(rows, pitch, P, probe_obs, bc, bc_pitch, status);
    return check_cuda(cudaGetLastError(), "novelty_bc_kernel");
}

extern "C" {

int cev_novelty_probe_obs_f32(cev_handle* h, const double* init, int64_t n, int seat, float* obs, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "novelty_probe_obs: null handle");
    CEV_REQUIRE(seat >= 0 && seat < 3, "novelty_probe_obs: seat must be 0, 1 or 2");
    CEV_REQUIRE(n >= 0, "novelty_probe_obs: n must be >= 0");
    if (n == 0) return CEV_OK;
    CEV_REQUIRE(init && obs, "novelty_probe_obs: null pointer");
    CEV_GUARD(h);
    novelty_probe_obs_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(init, n, seat, obs);
    return check_cuda(cudaGetLastError(), "novelty_probe_obs_kernel");
}

int cev_novelty_bc_f32(cev_handle* h, const float* rows, int64_t pitch, int in_dim, int64_t P, const float* probe_obs,
                       float* bc, int64_t bc_pitch, int32_t* status, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "novelty_bc: null handle");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "novelty_bc: in_dim must be 8 or 10");
    CEV_REQUIRE(P >= 0 && P <= 0x7FFFFFFFll, "novelty_bc: bad member count");
    if (P == 0) return CEV_OK;
    CEV_REQUIRE(rows && probe_obs && bc, "novelty_bc: null pointer");
    CEV_REQUIRE(pitch >= fc_offsets(in_dim).total && pitch % 4 == 0, "novelty_bc: bad pitch");
    CEV_REQUIRE(bc_pitch >= NV_BC, "novelty_bc: bc_pitch must be >= %d", NV_BC);
    CEV_REQUIRE(nv_aligned16(rows), "novelty_bc: rows must be 16-byte aligned");
    CEV_GUARD(h);
    cudaStream_t st = (cudaStream_t)stream;
    if (in_dim == IN_ADV) return launch_novelty_bc<IN_ADV>(h, rows, pitch, P, probe_obs, bc, bc_pitch, status, st);
    return launch_novelty_bc<IN_GOOD>(h, rows, pitch, P, probe_obs, bc, bc_pitch, status, st);
}

int cev_novelty_knn_f64(cev_handle* h, const float* bc, int64_t n, const float* ring, int64_t filled, int k,
                        double* novelty, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "novelty_knn: null handle");
    CEV_REQUIRE(k >= 1 && k <= CEV_NOVELTY_MAX_K, "novelty_knn: need 1 <= k <= %d, got %d", CEV_NOVELTY_MAX_K, k);
    CEV_REQUIRE(filled >= 1 && filled <= CEV_NOVELTY_MAX_ARCHIVE, "novelty_knn: need 1 <= filled <= %d",
                CEV_NOVELTY_MAX_ARCHIVE);
    CEV_REQUIRE(n >= 0, "novelty_knn: n must be >= 0");
    if (n == 0) return CEV_OK;
    CEV_REQUIRE(bc && ring && novelty, "novelty_knn: null pointer");
    CEV_GUARD(h);
    novelty_knn_kernel<<<(unsigned)((n + KN_WARPS - 1) / KN_WARPS), KN_WARPS * 32, 0, (cudaStream_t)stream>>>(
        bc, n, ring, (int)filled, k, novelty);
    return check_cuda(cudaGetLastError(), "novelty_knn_kernel");
}

}  // extern "C"
