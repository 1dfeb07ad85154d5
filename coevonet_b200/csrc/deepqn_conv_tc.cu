// K2, convolution stack on the 5th-generation tensor cores (implicit GEMM).
//
// Replaces the three convolutions + train-mode BatchNorm + ReLU of DeepQN.forward
// (Atari/deepqn.py:39-45: conv 8x8/4 (C -> 32), conv 4x4/2 (32 -> 64), conv 3x3/1 (64 -> 64); the "virtual
// batch norm" layers are BatchNorm2d in train mode at batch 1, SURVEY.md Appendix C #12, so the
// statistics are per FRAME over H x W).
//
// Each convolution is a per-member GEMM  Y[positions, Cout] = im2col(X)[positions, Cin*k*k] . W_m[Cout, Cin*k*k]^T:
//   conv1: 400 x (64 C) x 32     conv2: 81 x 512 x 64     conv3: 49 x 576 x 64     (per frame)
// One persistent CTA per SM, job = one frame; same warp roles as the rollout's opponent kernel
// (rollout_lockstep.cu): 8 producer warps, 1 TMA thread, 1 MMA thread, 4 epilogue warps.
//  * The job's input is staged in shared memory once: the u8 frame (conv1), or the previous layer's
//    pre-BatchNorm output with BatchNorm + ReLU applied on the way in (conv2, conv3: statistics per channel
//    over the frame's positions, two-pass, biased variance -- the normalisation is fused into the NEXT
//    layer's staging, so no activation round trip and no separate normalisation kernel between layers).
//  * Producers gather the im2col rows out of that copy (warp = 16-byte k chunk, lane = 4 output positions)
//    and write them, split into TF32 hi + lo, into the 128B-swizzled K-major A tiles.
//  * The member's conv weights [Cout x K] are already K-major: TMA streams [Cout x 32] boxes of the raw fp32
//    matrix through a 3-D tensor map (k, cout, member).  The raw tile IS the hi operand (the tensor core
//    reads an fp32 word truncated to TF32); the producers derive the lo tile (w - trunc(w), elementwise on
//    the swizzled bytes) next to it.
//  * tcgen05.mma kind::tf32, M = 128 positions, N = Cout, three MMAs per k-step (lo.hi + hi.lo + hi.hi =
//    3xTF32, fp32-level accuracy), accumulators double-buffered in TMEM; the epilogue adds the bias and stores
//    the pre-BatchNorm output [position][channel].
// A small kernel applies BatchNorm-3 + ReLU and writes conv3's output in torch's flatten order for the
// fully-connected stage (deepqn_tc.cu).
#include "deepqn_common.cuh"
#include "tc_common.cuh"

namespace cev {

constexpr int CV_THREADS = 448;                    // warps 0-3 epilogue, 4-11 producers, 12 TMA, 13 MMA
constexpr int CV_PROD = 256;
constexpr int CV_STAGES = 3;
constexpr int CV_BM = 128, CV_BK = 32;
constexpr uint32_t CV_A_BYTES = CV_BM * CV_BK * 4;  // 16 KB

template <int LAYER, int CIN_>
struct ConvGeo;
template <int CIN_>
struct ConvGeo<1, CIN_> {
    static constexpr int CIN = CIN_, KS = 8, STRIDE = 4, HIN = 84, HOUT = 20, COUT = 32;
    static constexpr size_t IN_BYTES = (size_t)CIN * 7056 + 1024;          // u8 frame + i/255 table
};
template <>
struct ConvGeo<2, 32> {
    static constexpr int CIN = 32, KS = 4, STRIDE = 2, HIN = 20, HOUT = 9, COUT = 64;
    static constexpr int LD = 401;                                          // padded channel row (400 positions)
    static constexpr size_t IN_BYTES = (size_t)CIN * LD * 4;
};
template <>
struct ConvGeo<3, 64> {
    static constexpr int CIN = 64, KS = 3, STRIDE = 1, HIN = 9, HOUT = 7, COUT = 64;
    static constexpr int LD = 82;                                           // 81 positions
    static constexpr size_t IN_BYTES = (size_t)CIN * LD * 4;
};

template <int LAYER, int CIN_>
struct ConvSmem {
    using G = ConvGeo<LAYER, CIN_>;
    static constexpr uint32_t B_BYTES = G::COUT * CV_BK * 4;                // 4 / 8 KB
    static constexpr uint32_t STAGE_BYTES = 2 * CV_A_BYTES + 2 * B_BYTES;    // A hi | A lo | B raw (= hi) | B lo
    static constexpr size_t off_in = (size_t)CV_STAGES * STAGE_BYTES;
    static constexpr size_t off_bar = (off_in + G::IN_BYTES + 15) & ~(size_t)15;
    static constexpr size_t total = off_bar + 256 + 1024 /*alignment slack*/;
    static_assert(total <= 232448, "conv stage does not fit the 227 KB of shared memory");
};

struct ConvParams {
    const float* members;
    int64_t pitch;
    int64_t n_frames;
    int B;                       // frames per member
    int w_off, b_off;            // this layer's weight / bias offsets in a member row
    int bn_g_off, bn_b_off;      // BatchNorm gamma / beta of the PREVIOUS layer (applied while staging)
    const uint8_t* frames;       // layer 1 input
    const float* y_in;           // layer 2, 3 input: previous pre-BatchNorm output [n_frames][positions][channels]
    float* y_out;                // [n_frames][positions][COUT]
};

template <int LAYER, int CIN_>
__global__ void __launch_bounds__(CV_THREADS, 1)
deepqn_conv_tc_kernel(const __grid_constant__ CUtensorMap map_w, const ConvParams p) {
    using G = ConvGeo<LAYER, CIN_>;
    using S = ConvSmem<LAYER, CIN_>;
    constexpr int NPOS = G::HOUT * G::HOUT;
    constexpr int NRT = (NPOS + CV_BM - 1) / CV_BM;            // row tiles per frame: 4, 1, 1
    constexpr int K = G::CIN * G::KS * G::KS;
    constexpr int NKT = K / CV_BK;                             // 8 (12), 16, 18
    static_assert(K % CV_BK == 0, "K must be a multiple of the k-tile");
    constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(G::COUT >> 3) << 17) |
                               ((uint32_t)(CV_BM >> 4) << 24);
    constexpr uint32_t TMEM_COLS = 128;

    extern __shared__ unsigned char cv_raw[];
    unsigned char* base = cv_raw + ((1024u - (tc_smem_u32(cv_raw) & 1023u)) & 1023u);   // stays in the shared space
    unsigned char* stage_mem = base;
    unsigned char* in_raw = base + S::off_in;
    uint64_t* bar_braw = reinterpret_cast<uint64_t*>(base + S::off_bar);   // [STAGES] raw B tile landed
    uint64_t* bar_full = bar_braw + CV_STAGES;                              // [STAGES] A + B lo written
    uint64_t* bar_empty = bar_full + CV_STAGES;                             // [STAGES] MMAs retired
    uint64_t* bar_tfull = bar_empty + CV_STAGES;                            // [2]
    uint64_t* bar_tempty = bar_tfull + 2;                                   // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < CV_STAGES; ++i) {
            tc_mbar_init(bar_braw + i, 1);
            tc_mbar_init(bar_full + i, CV_PROD / 32);
            tc_mbar_init(bar_empty + i, 1);
        }
        for (int i = 0; i < 2; ++i) {
            tc_mbar_init(bar_tfull + i, 1);
            tc_mbar_init(bar_tempty + i, 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 13) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tc_smem_u32(tmem_slot)),
                     "r"(TMEM_COLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp < 4) {
        // ===================== epilogue: + bias, store [position][channel] =====================
        const int q = warp;
        uint32_t pass = 0;
        for (int64_t f = blockIdx.x; f < p.n_frames; f += gridDim.x) {
            const float* bias = p.members + (f / p.B) * p.pitch + p.b_off;
            for (int rt = 0; rt < NRT; ++rt, ++pass) {
                const int pos = rt * CV_BM + q * 32 + lane;
                const uint32_t as = pass & 1, ause = pass >> 1;
                tc_mbar_wait(bar_tfull + as, ause & 1);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + as * G::COUT;
#pragma unroll
                for (int c0 = 0; c0 < G::COUT; c0 += 32) {
                    uint32_t v[32];
                    tmem_ld32(taddr + c0, v);
                    if (pos < NPOS) {
                        float4* dst = reinterpret_cast<float4*>(p.y_out + ((int64_t)f * NPOS + pos) * G::COUT + c0);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            dst[j] = make_float4(__uint_as_float(v[4 * j]) + __ldg(bias + c0 + 4 * j),
                                                 __uint_as_float(v[4 * j + 1]) + __ldg(bias + c0 + 4 * j + 1),
                                                 __uint_as_float(v[4 * j + 2]) + __ldg(bias + c0 + 4 * j + 2),
                                                 __uint_as_float(v[4 * j + 3]) + __ldg(bias + c0 + 4 * j + 3));
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                __syncwarp();
                if (lane == 0) tc_mbar_arrive(bar_tempty + as);
            }
        }
    } else if (warp < 12) {
        // ===================== producers: input staging (+ BatchNorm of the previous layer), im2col =====
        const int pt = threadIdx.x - 128;
        const int c = pt >> 5;                       // producer warp = 16-byte chunk (4 k) of every k-tile
        uint32_t it = 0;
        for (int64_t f = blockIdx.x; f < p.n_frames; f += gridDim.x) {
            const float* W = p.members + (f / p.B) * p.pitch;
            asm volatile("bar.sync 1, 256;\n" ::: "memory");      // every producer is done gathering from the old copy
            if constexpr (LAYER == 1) {
                uint8_t* in_u8 = in_raw;
                float* lut = reinterpret_cast<float*>(in_raw + (size_t)G::CIN * 7056);
                const uint4* src = reinterpret_cast<const uint4*>(p.frames + f * (int64_t)G::CIN * 7056);
                for (int i = pt; i < G::CIN * 7056 / 16; i += CV_PROD) reinterpret_cast<uint4*>(in_u8)[i] = __ldg(src + i);
                lut[pt] = __fdiv_rn((float)pt, 255.0f);           // bit-exact with the reference's x / 255
            } else {
                // previous layer's output [positions][channels] -> channel-major rows, BatchNorm + ReLU applied
                constexpr int NPIN = G::HIN * G::HIN;
                constexpr int CPW = G::CIN / 8;                    // channels per producer warp
                float* in_s = reinterpret_cast<float*>(in_raw);
                float gch[CPW], bch[CPW];                          // issued now, needed after the statistics
#pragma unroll
                for (int i = 0; i < CPW; ++i) {
                    gch[i] = __ldg(W + p.bn_g_off + c + 8 * i);
                    bch[i] = __ldg(W + p.bn_b_off + c + 8 * i);
                }
                const float4* src = reinterpret_cast<const float4*>(p.y_in + f * (int64_t)NPIN * G::CIN);
                for (int i = pt; i < NPIN * G::CIN / 4; i += CV_PROD) {
                    const float4 v = __ldg(src + i);
                    const int e = 4 * i, pos = e / G::CIN, c0 = e % G::CIN;
                    in_s[(c0 + 0) * G::LD + pos] = v.x;
                    in_s[(c0 + 1) * G::LD + pos] = v.y;
                    in_s[(c0 + 2) * G::LD + pos] = v.z;
                    in_s[(c0 + 3) * G::LD + pos] = v.w;
                }
                asm volatile("bar.sync 1, 256;\n" ::: "memory");
                // one warp per channel, two-pass statistics; the channels of a warp are independent chains,
                // unrolled so their shared-memory and shuffle latencies overlap.  The sums are of deviations from
                // the channel's first value: a constant channel then has exactly zero deviation and variance and
                // normalises to exactly beta (a rounded mean would leave ulps that rstd = 1/sqrt(eps) scales by 316)
                float mean[CPW], rstd[CPW], x0[CPW];
#pragma unroll
                for (int i = 0; i < CPW; ++i) {
                    const float* row = in_s + (c + 8 * i) * G::LD;
                    x0[i] = row[0];
                    float s1 = 0.f;
                    for (int q = lane; q < NPIN; q += 32) s1 += row[q] - x0[i];
                    mean[i] = s1;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                    for (int i = 0; i < CPW; ++i) mean[i] += __shfl_xor_sync(0xffffffffu, mean[i], o);
#pragma unroll
                for (int i = 0; i < CPW; ++i) {
                    const float* row = in_s + (c + 8 * i) * G::LD;
                    mean[i] = x0[i] + mean[i] * (1.0f / NPIN);
                    float qv = 0.f;
                    for (int q = lane; q < NPIN; q += 32) {
                        const float d = row[q] - mean[i];
                        qv = fmaf(d, d, qv);
                    }
                    rstd[i] = qv;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                    for (int i = 0; i < CPW; ++i) rstd[i] += __shfl_xor_sync(0xffffffffu, rstd[i], o);
#pragma unroll
                for (int i = 0; i < CPW; ++i) {
                    float* row = in_s + (c + 8 * i) * G::LD;
                    const float rs = 1.0f / sqrtf(rstd[i] * (1.0f / NPIN) + BN_EPS);
                    for (int q = lane; q < NPIN; q += 32) row[q] = fmaxf(fmaf((row[q] - mean[i]) * rs, gch[i], bch[i]), 0.f);
                }
            }
            asm volatile("bar.sync 1, 256;\n" ::: "memory");
            for (int rt = 0; rt < NRT; ++rt) {
                // this thread's four output positions and their top-left input offsets
                int ibase[4];
                bool valid[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int pos = rt * CV_BM + lane + 32 * j;
                    valid[j] = pos < NPOS;
                    const int pp = valid[j] ? pos : 0;
                    ibase[j] = (pp / G::HOUT) * G::STRIDE * G::HIN + (pp % G::HOUT) * G::STRIDE;
                }
                for (int kt = 0; kt < NKT; ++kt, ++it) {
                    const uint32_t st = it % CV_STAGES, use = it / CV_STAGES;
                    if (use > 0) tc_mbar_wait(bar_empty + st, (use - 1) & 1);
                    unsigned char* a_hi = stage_mem + (size_t)st * S::STAGE_BYTES;
                    unsigned char* a_lo = a_hi + CV_A_BYTES;
                    const int k0 = kt * CV_BK + 4 * c;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float x[4] = {0.f, 0.f, 0.f, 0.f};
                        if (valid[j]) {
                            if constexpr (LAYER == 1) {
                                const float* lut = reinterpret_cast<const float*>(in_raw + (size_t)G::CIN * 7056);
                                const int ci = k0 >> 6, ky = (k0 >> 3) & 7, kx0 = k0 & 7;
                                const uint32_t px = *reinterpret_cast<const uint32_t*>(
                                    in_raw + ci * 7056 + ibase[j] + ky * 84 + kx0);
                                x[0] = lut[px & 255u];
                                x[1] = lut[(px >> 8) & 255u];
                                x[2] = lut[(px >> 16) & 255u];
                                x[3] = lut[px >> 24];
                            } else if constexpr (LAYER == 2) {
                                const float* in_s = reinterpret_cast<const float*>(in_raw);
                                const int ci = k0 >> 4, ky = (k0 >> 2) & 3;
                                const float* src = in_s + ci * G::LD + ibase[j] + ky * G::HIN;
                                x[0] = src[0]; x[1] = src[1]; x[2] = src[2]; x[3] = src[3];
                            } else {
                                const float* in_s = reinterpret_cast<const float*>(in_raw);
#pragma unroll
                                for (int u = 0; u < 4; ++u) {
                                    const int k = k0 + u, ci = k / 9, rem = k - 9 * ci, ky = rem / 3, kx = rem - 3 * ky;
                                    x[u] = in_s[ci * G::LD + ibase[j] + ky * G::HIN + kx];
                                }
                            }
                        }
                        float hi[4], lo[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            hi[u] = __uint_as_float(__float_as_uint(x[u]) & 0xffffe000u);
                            lo[u] = x[u] - hi[u];
                        }
                        const int r = lane + 32 * j;
                        const int off = r * 128 + ((c ^ (r & 7)) << 4);
                        *reinterpret_cast<float4*>(a_hi + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
                        *reinterpret_cast<float4*>(a_lo + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
                    }
                    // the lo part of the weight tile, elementwise on the swizzled bytes TMA just landed
                    tc_mbar_wait(bar_braw + st, use & 1);
                    {
                        const float4* braw = reinterpret_cast<const float4*>(a_hi + 2 * CV_A_BYTES);
                        float4* blo = reinterpret_cast<float4*>(a_hi + 2 * CV_A_BYTES + S::B_BYTES);
                        for (int i = pt; i < (int)(S::B_BYTES / 16); i += CV_PROD) {
                            const float4 w = braw[i];
                            float4 l;
                            l.x = w.x - __uint_as_float(__float_as_uint(w.x) & 0xffffe000u);
                            l.y = w.y - __uint_as_float(__float_as_uint(w.y) & 0xffffe000u);
                            l.z = w.z - __uint_as_float(__float_as_uint(w.z) & 0xffffe000u);
                            l.w = w.w - __uint_as_float(__float_as_uint(w.w) & 0xffffe000u);
                            blo[i] = l;
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic writes -> tensor core reads
                    __syncwarp();
                    if (lane == 0) tc_mbar_arrive(bar_full + st);
                }
            }
        }
    } else if (warp == 12) {
        // ===================== TMA: the member's conv weights, [COUT x 32] boxes =====================
        if (lane == 0) {
            uint32_t it = 0;
            for (int64_t f = blockIdx.x; f < p.n_frames; f += gridDim.x) {
                const int m = (int)(f / p.B);
                for (int rt = 0; rt < NRT; ++rt)
                    for (int kt = 0; kt < NKT; ++kt, ++it) {
                        const uint32_t st = it % CV_STAGES, use = it / CV_STAGES;
                        if (use > 0) tc_mbar_wait(bar_empty + st, (use - 1) & 1);
                        unsigned char* braw = stage_mem + (size_t)st * S::STAGE_BYTES + 2 * CV_A_BYTES;
                        tc_mbar_expect_tx(bar_braw + st, S::B_BYTES);
                        tma_load_3d(braw, &map_w, bar_braw + st, kt * CV_BK, 0, m);
                    }
            }
        }
    } else {
        // ===================== MMA issuer =====================
        const uint32_t stage_base = tc_smem_u32(stage_mem);
        uint32_t it = 0, pass = 0;
        for (int64_t f = blockIdx.x; f < p.n_frames; f += gridDim.x)
            for (int rt = 0; rt < NRT; ++rt, ++pass) {
                const uint32_t as = pass & 1, ause = pass >> 1;
                if (ause > 0) tc_mbar_wait(bar_tempty + as, (ause - 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t d_tmem = tmem_base + as * G::COUT;
                for (int kt = 0; kt < NKT; ++kt, ++it) {
                    const uint32_t st = it % CV_STAGES, use = it / CV_STAGES;
                    tc_mbar_wait(bar_full + st, use & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    {
                        // issued by one elected lane of the converged warp (tc_issue_ktile_3xtf32): with N = 32 / 64 an
                        // MMA occupies the tensor pipe ~45 cycles, a divergent `if (lane == 0)` issue costs ~130
                        const uint32_t s_addr = stage_base + st * S::STAGE_BYTES;
                        tc_issue_ktile_3xtf32(d_tmem, umma_desc_sw128(s_addr), umma_desc_sw128(s_addr + CV_A_BYTES),
                                              umma_desc_sw128(s_addr + 2 * CV_A_BYTES),
                                              umma_desc_sw128(s_addr + 2 * CV_A_BYTES + S::B_BYTES), IDESC, kt ? 1u : 0u,
                                              tc_smem_u32(bar_empty + st));
                        if (kt == NKT - 1) tc_commit_elected(tc_smem_u32(bar_tfull + as));
                    }
                    __syncwarp();
                }
            }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 13) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
    }
}

// BatchNorm-3 + ReLU on conv3's output [49][64] and torch's flatten order (x.reshape(B, -1) of [C, H, W]:
// index c * 49 + pos).  One CTA per frame, thread = channel.
__global__ void __launch_bounds__(64) deepqn_bn3_flatten_kernel(const float* __restrict__ y3, int64_t n_frames, int B,
                                                                const float* __restrict__ members, int64_t pitch,
                                                                int g_off, int b_off, float* __restrict__ act3) {
    const int ch = threadIdx.x;
    for (int64_t f = blockIdx.x; f < n_frames; f += gridDim.x) {
        const float* src = y3 + f * 49 * 64 + ch;
        float v[49];
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 49; ++i) v[i] = src[i * 64];
#pragma unroll
        for (int i = 0; i < 49; ++i) s += v[i] - v[0];          // deviations: exact zero for a constant channel
        const float mean = v[0] + s * (1.0f / 49);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 49; ++i) {
            const float d = v[i] - mean;
            q = fmaf(d, d, q);
        }
        const float rstd = 1.0f / sqrtf(q * (1.0f / 49) + BN_EPS);
        const float* W = members + (f / B) * pitch;
        const float g = __ldg(W + g_off + ch), b = __ldg(W + b_off + ch);
        float* dst = act3 + f * 3136 + ch * 49;
#pragma unroll
        for (int i = 0; i < 49; ++i) dst[i] = fmaxf(fmaf((v[i] - mean) * rstd, g, b), 0.f);
    }
}

template <int LAYER, int CIN_>
static int launch_conv_layer(cev_handle* h, EncodeTiledFn encode, const float* members, int64_t pitch, int P,
                             const ConvParams& p, cudaStream_t stream) {
    using G = ConvGeo<LAYER, CIN_>;
    using S = ConvSmem<LAYER, CIN_>;
    constexpr int K = G::CIN * G::KS * G::KS;
    CUtensorMap map_w;
    cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)G::COUT, (cuuint64_t)P};
    cuuint64_t strides[2] = {(cuuint64_t)K * 4, (cuuint64_t)pitch * 4};
    cuuint32_t box[3] = {CV_BK, (cuuint32_t)G::COUT, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode(&map_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(members + p.w_off), dims, strides,
                        box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("deepqn_conv_tc: cuTensorMapEncodeTiled(conv%d weights) failed with %d", LAYER, (int)r);
        return CEV_ERR_CUDA;
    }
    auto kern = deepqn_conv_tc_kernel<LAYER, CIN_>;
    CEV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::total));
    const int64_t grid = p.n_frames < h->n_sm ? p.n_frames : h->n_sm;
    kern<<<(unsigned)grid, CV_THREADS, S::total, stream>>>(map_w, p);
    return check_cuda(cudaGetLastError(), "deepqn_conv_tc_kernel");
}

int launch_deepqn_conv_tc(cev_handle* h, const float* members, int64_t pitch, int P, int B, int c_in, int n_act,
                          const uint8_t* frames, float* y1, float* y2, float* y3, float* act3, cudaStream_t stream) {
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) {
        set_error("deepqn_conv_tc: cuTensorMapEncodeTiled is not available from the driver");
        return CEV_ERR_UNSUPPORTED;
    }
    const DqnOffsets o = dqn_offsets(c_in, n_act);
    ConvParams p{};
    p.members = members;
    p.pitch = pitch;
    p.n_frames = (int64_t)P * B;
    p.B = B;
    int rc;
    // conv1: u8 frame -> y1 [400][32]
    p.w_off = o.c1w;
    p.b_off = o.c1b;
    p.frames = frames;
    p.y_in = nullptr;
    p.y_out = y1;
    rc = c_in == 4 ? launch_conv_layer<1, 4>(h, encode, members, pitch, P, p, stream)
                   : launch_conv_layer<1, 6>(h, encode, members, pitch, P, p, stream);
    if (rc) return rc;
    // conv2: BatchNorm-1 + ReLU while staging y1 -> y2 [81][64]
    p.w_off = o.c2w;
    p.b_off = o.c2b;
    p.bn_g_off = o.bn1g;
    p.bn_b_off = o.bn1b;
    p.frames = nullptr;
    p.y_in = y1;
    p.y_out = y2;
    rc = launch_conv_layer<2, 32>(h, encode, members, pitch, P, p, stream);
    if (rc) return rc;
    // conv3: BatchNorm-2 + ReLU while staging y2 -> y3 [49][64]
    p.w_off = o.c3w;
    p.b_off = o.c3b;
    p.bn_g_off = o.bn2g;
    p.bn_b_off = o.bn2b;
    p.y_in = y2;
    p.y_out = y3;
    rc = launch_conv_layer<3, 64>(h, encode, members, pitch, P, p, stream);
    if (rc) return rc;
    const int64_t grid = p.n_frames < 4096 ? p.n_frames : 4096;
    deepqn_bn3_flatten_kernel<<<(unsigned)grid, 64, 0, stream>>>(y3, p.n_frames, B, members, pitch, o.bn3g, o.bn3b, act3);
    return check_cuda(cudaGetLastError(), "deepqn_bn3_flatten_kernel");
}

}  // namespace cev
