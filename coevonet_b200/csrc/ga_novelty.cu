// Co-GA novelty search (Lehman & Stanley 2011; Such et al. 2017): the k-nearest-neighbour novelty of a GA
// population's behaviour characterisations against the whole population plus an archive
// (cev_ga_novelty_knn_f64), and the archive draws (cev_ga_novelty_draw_i64).  A translation unit of its own:
// ptxas allocates the registers of the kernels of one module together, so every existing kernel keeps its SASS.
//
// The k-NN is the hot path: n members x (P + filled) candidates x 160 dimensions per role and generation.  A CTA
// takes a tile of GN_BM members and a range of candidate tiles (a split, blockIdx.y).  Per candidate tile of GN_BN
// rows, each thread accumulates an 8 x 8 register tile of squared distances in fp32 (FADD + FFMA, the dimensions
// in order), the tile's distances go to shared memory, and one warp per member absorbs them into the member's
// sorted list of the k smallest (distance, index) keys.  A merge kernel combines the splits' lists and forms the
// novelty.  The k smallest keys of a total order do not depend on the tiling or on the split, so neither does a
// member's novelty.
#include <algorithm>

#include "common.cuh"

namespace cev {

constexpr int GN_D = CEV_NOVELTY_BC_DIM;      // 160 floats per characterisation
constexpr int GN_BM = 128;                    // members per CTA tile
constexpr int GN_BN = 128;                    // candidates per tile
constexpr int GN_T = 256;                     // threads: 16 x 16, each an 8 x 8 tile of pairs
constexpr int GN_DK = 32;                     // dimensions per staged candidate chunk
constexpr int GN_XLD = GN_BM + 4;             // Xs[t][m]: the member tile, transposed, resident
constexpr int GN_CLD = GN_BN + 4;             // Cs[t][c]: one chunk of the candidate tile, transposed
constexpr int GN_DLD = GN_BN + 4;             // Ds[m][c]: the tile's distances
constexpr int GN_LD = 32;                     // keys per member list (k <= 32)
constexpr int GN_MPW = GN_BM / (GN_T / 32);   // members absorbed per warp
constexpr int GN_CHUNKS = GN_D / GN_DK;
constexpr unsigned long long GN_NONE = ~0ull; // the empty list entry: above every key
static_assert(GN_D % GN_DK == 0 && GN_DK % 4 == 0, "chunking");
static_assert(GN_BN * GN_DK / 4 == 4 * GN_T, "four float4 loads per thread per chunk");
static_assert(GN_LD == CEV_NOVELTY_MAX_K, "one lane per list entry");
constexpr size_t GN_SMEM = (size_t)(GN_D * GN_XLD + GN_DK * GN_CLD + GN_BM * GN_DLD) * sizeof(float) +
                           (size_t)GN_BM * GN_LD * sizeof(unsigned long long);

// Sort key of (distance, candidate index): distances are +0 .. +inf or NaN (a sum of squares from +0), so the fp32
// bit pattern orders them; every NaN maps to 0x7fffffff, above +inf.  Keys are unique (the index is).
__device__ __forceinline__ unsigned long long gn_key(float d, uint32_t c) {
    const uint32_t b = isnan(d) ? 0x7fffffffu : __float_as_uint(d);
    return ((unsigned long long)b << 32) | c;
}

__device__ __forceinline__ unsigned long long gn_shfl(unsigned long long v, int src) {
    return __shfl_sync(0xffffffffu, v, src);
}

// Insert the lanes' candidate keys `ck` into the warp's sorted list (lane l holds the l-th smallest key): the
// candidates below the k-th key are inserted one at a time, in lane order.
__device__ __forceinline__ void gn_absorb(unsigned long long& key, unsigned long long ck, int k, int lane) {
    unsigned cand = __ballot_sync(0xffffffffu, ck < gn_shfl(key, k - 1));
    while (cand) {
        const int src = __ffs(cand) - 1;
        cand &= cand - 1;
        const unsigned long long v = gn_shfl(ck, src);
        if (v >= gn_shfl(key, k - 1)) continue;                   // no longer among the k smallest
        const int pos = __ffs(__ballot_sync(0xffffffffu, v < key)) - 1;
        const unsigned long long up = __shfl_up_sync(0xffffffffu, key, 1);
        if (lane > pos) key = up;
        else if (lane == pos) key = v;
    }
}

struct GnArgs {
    const float* x;          // members [n][x_pitch]
    int64_t x_pitch, n, row0;
    const float* pop;        // gathered population [P][pop_pitch]
    int64_t pop_pitch, P;
    const float* ring;       // archive [>= filled][160]
    int64_t filled;
    int k, n_tiles, splits;
    unsigned long long* part;  // [splits][n][k]
};

__device__ __forceinline__ const float* gn_cand_row(const GnArgs& a, int64_t c) {
    return c < a.P ? a.pop + c * a.pop_pitch : a.ring + (c - a.P) * GN_D;
}

__global__ void __launch_bounds__(GN_T, 1) ga_novelty_knn_kernel(const GnArgs a) {
    extern __shared__ float4 gn_smem[];
    float* Xs = reinterpret_cast<float*>(gn_smem);
    float* Cs = Xs + GN_D * GN_XLD;
    float* Ds = Cs + GN_DK * GN_CLD;
    unsigned long long* Ls = reinterpret_cast<unsigned long long*>(Ds + GN_BM * GN_DLD);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid & 15, ty = tid >> 4;
    const int64_t i0 = (int64_t)blockIdx.x * GN_BM;
    const int64_t total = a.P + a.filled;
    const int s = blockIdx.y;
    const int64_t tb = (int64_t)a.n_tiles * s / a.splits, te = (int64_t)a.n_tiles * (s + 1) / a.splits;

    // ---- the member tile, transposed, and the empty lists --------------------------------------------------
    for (int idx = tid; idx < GN_BM * GN_D / 4; idx += GN_T) {
        const int m = idx / (GN_D / 4), q = idx - m * (GN_D / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i0 + m < a.n) v = __ldg(reinterpret_cast<const float4*>(a.x + (i0 + m) * a.x_pitch) + q);
        Xs[(4 * q + 0) * GN_XLD + m] = v.x;
        Xs[(4 * q + 1) * GN_XLD + m] = v.y;
        Xs[(4 * q + 2) * GN_XLD + m] = v.z;
        Xs[(4 * q + 3) * GN_XLD + m] = v.w;
    }
    for (int idx = tid; idx < GN_BM * GN_LD; idx += GN_T) Ls[idx] = GN_NONE;

    // ---- candidate chunks, one step = (tile, 32 dimensions), the next step's loads in registers ----------------
    float4 pf[4];
    auto load = [&](int64_t step) {
        const int64_t c0 = (tb + step / GN_CHUNKS) * GN_BN;
        const int d0 = (int)(step % GN_CHUNKS) * GN_DK;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int idx = tid + r * GN_T, c = idx >> 3, q = idx & 7;
            pf[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (c0 + c < total) pf[r] = __ldg(reinterpret_cast<const float4*>(gn_cand_row(a, c0 + c) + d0) + q);
        }
    };
    const int64_t n_steps = (te - tb) * GN_CHUNKS;
    if (n_steps > 0) load(0);
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    for (int64_t step = 0; step < n_steps; ++step) {
        __syncthreads();                                 // the previous chunk is consumed
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int idx = tid + r * GN_T, c = idx >> 3, q = idx & 7;
            Cs[(4 * q + 0) * GN_CLD + c] = pf[r].x;
            Cs[(4 * q + 1) * GN_CLD + c] = pf[r].y;
            Cs[(4 * q + 2) * GN_CLD + c] = pf[r].z;
            Cs[(4 * q + 3) * GN_CLD + c] = pf[r].w;
        }
        __syncthreads();
        if (step + 1 < n_steps) load(step + 1);
        const int d0 = (int)(step % GN_CHUNKS) * GN_DK;
        // thread (ty, tx): members ty*4 + i and 64 + ty*4 + i, candidates tx*4 + j and 64 + tx*4 + j
#pragma unroll 4
        for (int t = 0; t < GN_DK; ++t) {
            const float* xr = Xs + (d0 + t) * GN_XLD;
            const float* cr = Cs + t * GN_CLD;
            const float4 x0 = *reinterpret_cast<const float4*>(xr + 4 * ty);
            const float4 x1 = *reinterpret_cast<const float4*>(xr + 64 + 4 * ty);
            const float4 c0 = *reinterpret_cast<const float4*>(cr + 4 * tx);
            const float4 c1 = *reinterpret_cast<const float4*>(cr + 64 + 4 * tx);
            const float xm[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
            const float cc[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float e = __fsub_rn(xm[i], cc[j]);
                    acc[i][j] = fmaf(e, e, acc[i][j]);
                }
        }
        if (step % GN_CHUNKS != GN_CHUNKS - 1) continue;
        // ---- the tile is complete: distances to shared memory, then one warp per member absorbs them -----------
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int m = (i < 4 ? 0 : 64) + 4 * ty + (i & 3);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float4 d;
                d.x = __fsqrt_rn(acc[i][4 * h + 0]);
                d.y = __fsqrt_rn(acc[i][4 * h + 1]);
                d.z = __fsqrt_rn(acc[i][4 * h + 2]);
                d.w = __fsqrt_rn(acc[i][4 * h + 3]);
                *reinterpret_cast<float4*>(Ds + m * GN_DLD + 64 * h + 4 * tx) = d;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
        }
        __syncthreads();
        const int64_t c0 = (tb + step / GN_CHUNKS) * GN_BN;
        for (int mm = 0; mm < GN_MPW; ++mm) {
            const int m = warp * GN_MPW + mm;
            const int64_t gi = i0 + m;
            if (gi >= a.n) break;                                    // warp-uniform
            unsigned long long key = Ls[m * GN_LD + lane];
#pragma unroll
            for (int r = 0; r < GN_BN / 32; ++r) {
                const int64_t c = c0 + r * 32 + lane;
                const bool valid = c < total && c != a.row0 + gi;   // excluded by id, not by value
                const unsigned long long ck = valid ? gn_key(Ds[m * GN_DLD + r * 32 + lane], (uint32_t)c) : GN_NONE;
                gn_absorb(key, ck, a.k, lane);
            }
            Ls[m * GN_LD + lane] = key;
        }
    }
    __syncthreads();
    // ---- this split's lists ---------------------------------------------------------------------------------
    for (int mm = 0; mm < GN_MPW; ++mm) {
        const int m = warp * GN_MPW + mm;
        const int64_t gi = i0 + m;
        if (gi >= a.n) break;
        if (lane < a.k) a.part[((int64_t)s * a.n + gi) * a.k + lane] = Ls[m * GN_LD + lane];
    }
}

// One warp per member: the k smallest keys over the splits' lists, then N = (fp64 sum of the k_eff smallest
// distances, in key order, from +0) / k_eff.
__global__ void __launch_bounds__(256) ga_novelty_merge_kernel(const unsigned long long* __restrict__ part,
                                                              int64_t n, int splits, int k, int k_eff,
                                                              double* __restrict__ novelty) {
    const int lane = threadIdx.x & 31;
    const int64_t i = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (i >= n) return;                                             // warp-uniform
    unsigned long long key = GN_NONE;
    for (int s = 0; s < splits; ++s) {
        const unsigned long long ck = lane < k ? part[((int64_t)s * n + i) * k + lane] : GN_NONE;
        gn_absorb(key, ck, k, lane);
    }
    double sum = 0.0;
    for (int j = 0; j < k_eff; ++j)
        sum = __dadd_rn(sum, (double)__uint_as_float((uint32_t)(gn_shfl(key, j) >> 32)));
    if (lane == 0) novelty[i] = __ddiv_rn(sum, (double)k_eff);
}

// Archive draw j: word (j & 3) of Philox(seed; (j >> 2, 0, gen, role | CEV_KIND_GA_NOVELTY << 8)), scaled to [0, P)
__global__ void __launch_bounds__(256) ga_novelty_draw_kernel(uint32_t k0, uint32_t k1, uint32_t gen, int role,
                                                             int m, uint64_t P, int64_t* __restrict__ out) {
    const int j = blockIdx.x * 256 + threadIdx.x;
    if (j >= m) return;
    const U4 v = philox4x32_10(U4{(uint32_t)(j >> 2), 0u, gen, noise_tag(CEV_KIND_GA_NOVELTY, role)}, k0, k1);
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    out[j] = (int64_t)(((uint64_t)w[j & 3] * P) >> 32);
}

}  // namespace cev

using namespace cev;

static bool gn_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

extern "C" {

int cev_ga_novelty_knn_f64(cev_handle* h, const float* x, int64_t x_pitch, int64_t n, int64_t row0, const float* pop,
                           int64_t pop_pitch, int64_t P, const float* ring, int64_t filled, int k, int splits,
                           double* novelty, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "ga_novelty_knn: null handle");
    CEV_REQUIRE(k >= 1 && k <= CEV_NOVELTY_MAX_K, "ga_novelty_knn: need 1 <= k <= %d, got %d", CEV_NOVELTY_MAX_K, k);
    CEV_REQUIRE(P >= 1 && P <= 0x7FFFFFFFll, "ga_novelty_knn: need 1 <= P < 2^31");
    CEV_REQUIRE(filled >= 0 && filled <= CEV_NOVELTY_MAX_ARCHIVE, "ga_novelty_knn: need 0 <= filled <= %d",
                CEV_NOVELTY_MAX_ARCHIVE);
    CEV_REQUIRE(P - 1 + filled >= 1, "ga_novelty_knn: a member needs at least one other candidate");
    CEV_REQUIRE(n >= 0 && row0 >= 0 && row0 + n <= P, "ga_novelty_knn: need 0 <= row0 <= row0 + n <= P");
    CEV_REQUIRE(splits >= 0, "ga_novelty_knn: splits must be >= 0 (0 = automatic)");
    if (n == 0) return CEV_OK;
    CEV_REQUIRE(x && pop && novelty && (ring || filled == 0), "ga_novelty_knn: null pointer");
    CEV_REQUIRE(x_pitch >= GN_D && x_pitch % 4 == 0 && pop_pitch >= GN_D && pop_pitch % 4 == 0,
                "ga_novelty_knn: row pitches must be multiples of 4 floats >= %d", GN_D);
    CEV_REQUIRE(gn_aligned16(x) && gn_aligned16(pop) && (filled == 0 || gn_aligned16(ring)),
                "ga_novelty_knn: characterisations must be 16-byte aligned");
    CEV_GUARD(h);
    const int64_t m_tiles = (n + GN_BM - 1) / GN_BM;
    const int64_t n_tiles = (P + filled + GN_BN - 1) / GN_BN;
    CEV_REQUIRE(m_tiles <= 0x7FFFFFFFll, "ga_novelty_knn: too many members");
    // automatic: at least 8 waves of the 1-CTA-per-SM kernel where the candidates allow it (the last wave's tail
    // then costs at most an eighth)
    int64_t S = splits ? splits : (8ll * h->n_sm + m_tiles - 1) / m_tiles;
    S = std::max<int64_t>(1, std::min<int64_t>({S, n_tiles, 65535}));
    const size_t need = (size_t)S * n * k * sizeof(unsigned long long);
    if (h->workspace_bytes < need) {
        if (h->workspace) cudaFree(h->workspace);
        h->workspace = nullptr;
        h->workspace_bytes = 0;
        CEV_CUDA(cudaMalloc(&h->workspace, need));
        h->workspace_bytes = need;
    }
    static bool configured[16] = {};
    if (h->device >= 16 || !configured[h->device]) {
        CEV_CUDA(cudaFuncSetAttribute(ga_novelty_knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)GN_SMEM));
        if (h->device < 16) configured[h->device] = true;
    }
    GnArgs a{x, x_pitch, n, row0, pop, pop_pitch, P, ring, filled, k, (int)n_tiles, (int)S,
             static_cast<unsigned long long*>(h->workspace)};
    cudaStream_t st = (cudaStream_t)stream;
    ga_novelty_knn_kernel<<<dim3((unsigned)m_tiles, (unsigned)S), GN_T, GN_SMEM, st>>>(a);
    CEV_CUDA(cudaGetLastError());
    const int k_eff = (int)std::min<int64_t>(k, P - 1 + filled);
    ga_novelty_merge_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(a.part, n, (int)S, k, k_eff, novelty);
    return check_cuda(cudaGetLastError(), "ga_novelty_merge_kernel");
}

int cev_ga_novelty_draw_i64(cev_handle* h, uint64_t seed, uint32_t gen, int role, int m, int64_t P, int64_t* out,
                            cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "ga_novelty_draw: null handle");
    CEV_REQUIRE(role >= 0 && role < 256, "ga_novelty_draw: role must be in [0, 256)");
    CEV_REQUIRE(m >= 0, "ga_novelty_draw: m must be >= 0");
    CEV_REQUIRE(P >= 1 && P <= 0x100000000ll, "ga_novelty_draw: need 1 <= P <= 2^32");
    if (m == 0) return CEV_OK;
    CEV_REQUIRE(out != nullptr, "ga_novelty_draw: null pointer");
    CEV_GUARD(h);
    ga_novelty_draw_kernel<<<(unsigned)((m + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        (uint32_t)(seed & 0xFFFFFFFFull), (uint32_t)(seed >> 32), gen, role, m, (uint64_t)P, out);
    return check_cuda(cudaGetLastError(), "ga_novelty_draw_kernel");
}

}  // extern "C"
