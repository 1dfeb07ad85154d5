// K2, fully-connected stage on the 5th-generation tensor cores, fp32-accurate (3xTF32).
//
// fc1 of DeepQN (Atari/deepqn.py:27,46: 3136 -> 512) holds 95 % of a member's bytes and is a dense
// contraction: per member  H[512, frames] = W1[512, 3136] . X[frames, 3136]^T.  The stage is HBM bound
// (6.4 MB of W1 per member, read once), so the tensor pipe has time to spare: every product is issued three
// times (lo.hi + hi.lo + hi.hi, "3xTF32": fp32-level accuracy, logits within 2e-5 of the reference's fp32
// forward) -- affordable because the WEIGHTS are the M-side operand (M = 128 rows of W1 per MMA, four row
// tiles) and the frames the N side (N = 16): an MMA is 128 x 16 x 8 instead of the 128-frame-row form whose M
// was 127/128 padding at one frame per member.
//
// One persistent CTA per SM, job = member.  Per k-tile of 32:
//   warp 0      TMA: the raw W1 tile [256 rows x 32 k] (3-D tensor map (k, row, member), 128B swizzle) and the
//               raw activation tile [16 frames x 32 k] into a 4-slot ring
//   warps 2-5   derive the lo parts: hi = the raw fp32 word as the tensor core reads it (truncated to TF32),
//               lo = w - trunc(w).  W1 lo goes to TENSOR MEMORY (tcgen05.st, lane = W1 row, 32 columns per row
//               tile and k-tile, two slots): the MMA takes it as a TMEM A operand, so it never costs shared-memory
//               bandwidth -- with lo tiles in shared memory the stage moved 168 KB per k-tile through the 128 B/clk
//               shared-memory port (TMA write + LDS + STS + two operand fetches) and was bound by it, not by HBM.
//               The activations' lo tile goes right behind their hi tile, so [x_hi | x_lo] is ONE 32-row N operand.
//   warp 1      16 x tcgen05.mma.cta_group::1.kind::tf32 (2 row tiles x 4 k-steps x {w_hi (smem) . [x_hi | x_lo]
//               (N = 32), w_lo (TMEM) . x_hi (N = 16)}) into three accumulator column groups that the epilogue adds
//   warps 6-9   epilogue per 256-row pass: tcgen05.ld, bias + ReLU into shared memory, then the 512 -> A output
//               layer (Atari/deepqn.py:47) accumulated in registers over the two passes, first-max argmax.
// Frames are processed 16 at a time (W1 is re-streamed for every further block of 16 frames of a member).
#include <stdlib.h>

#include "tc_common.cuh"

namespace cev {

constexpr int F3_THREADS = 320;
constexpr int F3_BK = 32;                       // fp32 per k-tile = 128 bytes = one swizzle row
constexpr int F3_K = 3136;
constexpr int F3_KT = F3_K / F3_BK;             // 98 k-tiles
constexpr int F3_ROWS = 256;                    // W1 rows per pass = two M tiles of 128
constexpr int F3_NPASS = 512 / F3_ROWS;
constexpr int F3_NB = 16;                       // frames per block = MMA N
constexpr int F3_R = 5, F3_L = 4;               // raw slots (shared memory), W1-lo slots (tensor memory)
constexpr uint32_t F3_A_BYTES = F3_ROWS * F3_BK * 4;          // 32 KB
constexpr uint32_t F3_X_BYTES = F3_NB * F3_BK * 4;            // 2 KB
constexpr uint32_t F3_SLOT = F3_A_BYTES + 2 * F3_X_BYTES;     // raw slot: W1 raw | x hi (raw) | x lo = 36 KB
constexpr size_t F3_OFF_HS = (size_t)F3_R * F3_SLOT;
constexpr int F3_MAX_ACT = 32;
// hs: [256][16] fp32 = 16 KB; the logits exchange [A][16] reuses its head once the last pass has been consumed
constexpr size_t F3_OFF_BAR = F3_OFF_HS + (size_t)F3_ROWS * F3_NB * 4;
constexpr size_t F3_SMEM = F3_OFF_BAR + 256 + 1024 /*alignment*/;
constexpr int F3_ACC = 3 * F3_NB;                             // accumulator columns per row tile: hh | hl | lh
constexpr int F3_TM_LO = 2 * 2 * F3_ACC;                      // first TMEM column of the W1-lo slots (after the accumulators)
constexpr int F3_TM_LSLOT = 2 * F3_BK;                        // columns per lo slot: 2 row tiles x 32 k
static_assert(F3_TM_LO + F3_L * F3_TM_LSLOT <= 512, "tensor memory budget");
static_assert(F3_SLOT % 1024 == 0, "slots must keep the 1024-byte alignment of the swizzle atoms");
static_assert(F3_SMEM <= 232448, "fc stage exceeds the 227 KB shared-memory limit");

// instruction descriptors: D = F32, A = B = TF32, both K-major, M = 128, N = 32 / 16
constexpr uint32_t F3_IDESC32 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)((2 * F3_NB) >> 3) << 17) |
                                ((uint32_t)(128 >> 4) << 24);
constexpr uint32_t F3_IDESC16 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(F3_NB >> 3) << 17) |
                                ((uint32_t)(128 >> 4) << 24);

struct TcParams {
    const float* members;
    int64_t pitch;
    int P, B, n_act;
    int f1b_off, ow_off, ob_off;
    float* logits;
    int32_t* actions;
};

__global__ void __launch_bounds__(F3_THREADS, 1)
deepqn_fc_tc_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w,
                    const TcParams p) {
    extern __shared__ unsigned char f3_raw[];
    unsigned char* base = f3_raw + ((1024u - (tc_smem_u32(f3_raw) & 1023u)) & 1023u);
    unsigned char* raw_mem = base;                                   // R x (W1 raw | x raw | x lo)
    float* hs = reinterpret_cast<float*>(base + F3_OFF_HS);          // [256 rows][16 frames], 16B chunks swizzled
    float* lgs = hs;                                                 // [A][16], after the last pass
    uint64_t* bar_raw_full = reinterpret_cast<uint64_t*>(base + F3_OFF_BAR);
    uint64_t* bar_raw_empty = bar_raw_full + F3_R;
    uint64_t* bar_lo_full = bar_raw_empty + F3_R;
    uint64_t* bar_lo_empty = bar_lo_full + F3_L;
    uint64_t* bar_tfull = bar_lo_empty + F3_L;        // [2] accumulators of a pass ready
    uint64_t* bar_tempty = bar_tfull + 2;             // [2] accumulators drained
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar_tempty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_fblk = (p.B + F3_NB - 1) / F3_NB;

    if (threadIdx.x == 0) {
        for (int i = 0; i < F3_R; ++i) {
            tc_mbar_init(bar_raw_full + i, 1);
            tc_mbar_init(bar_raw_empty + i, 1);
        }
        for (int i = 0; i < F3_L; ++i) {
            tc_mbar_init(bar_lo_full + i, 4);          // one arrive per lo-producer warp
            tc_mbar_init(bar_lo_empty + i, 1);
        }
        for (int i = 0; i < 2; ++i) {
            tc_mbar_init(bar_tfull + i, 1);
            tc_mbar_init(bar_tempty + i, 4);           // one arrive per epilogue warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        // 2 (ping-pong) x 2 (row tiles) x 48 accumulator columns = 192, then 2 W1-lo slots x 64 columns = 320 -> 512
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(tc_smem_u32(tmem_slot)),
                     "r"(512u)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA: raw W1 tile + raw activation tile =====================
        if (lane == 0) {
            uint32_t it = 0;
            for (int m = blockIdx.x; m < p.P; m += gridDim.x)
                for (int fb = 0; fb < n_fblk; ++fb)
                    for (int ps = 0; ps < F3_NPASS; ++ps)
                        for (int kt = 0; kt < F3_KT; ++kt, ++it) {
                            const uint32_t rs = it % F3_R, use = it / F3_R;
                            if (use > 0) tc_mbar_wait(bar_raw_empty + rs, (use - 1) & 1);
                            unsigned char* a = raw_mem + (size_t)rs * F3_SLOT;
                            tc_mbar_expect_tx(bar_raw_full + rs, F3_A_BYTES + F3_X_BYTES);
                            tma_load_3d(a, &map_w, bar_raw_full + rs, kt * F3_BK, ps * F3_ROWS, m);
                            tma_load_2d(a + F3_A_BYTES, &map_x, bar_raw_full + rs, kt * F3_BK, m * p.B + fb * F3_NB);
                        }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        uint32_t it = 0, pass = 0;
        for (int m = blockIdx.x; m < p.P; m += gridDim.x)
            for (int fb = 0; fb < n_fblk; ++fb)
                for (int ps = 0; ps < F3_NPASS; ++ps, ++pass) {
                    const uint32_t as = pass & 1, ause = pass >> 1;
                    if (ause > 0) tc_mbar_wait(bar_tempty + as, (ause - 1) & 1);      // epilogue drained it
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint32_t d_tmem = tmem_base + as * (2 * F3_ACC);
                    for (int kt = 0; kt < F3_KT; ++kt, ++it) {
                        const uint32_t rs = it % F3_R, ruse = it / F3_R, ls = it % F3_L, luse = it / F3_L;
                        tc_mbar_wait(bar_raw_full + rs, ruse & 1);
                        tc_mbar_wait(bar_lo_full + ls, luse & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                        if (lane == 0) {
                            const uint32_t hi_addr = tc_smem_u32(raw_mem + (size_t)rs * F3_SLOT);
                            const uint32_t lo_tmem = tmem_base + F3_TM_LO + ls * F3_TM_LSLOT;
                            const uint64_t x_hilo = umma_desc_sw128(hi_addr + F3_A_BYTES);    // 32 rows: x hi | x lo
#pragma unroll
                            for (int t = 0; t < 2; ++t) {
                                const uint64_t w_hi = umma_desc_sw128(hi_addr + t * (128 * F3_BK * 4));
#pragma unroll
                                for (int k8 = 0; k8 < F3_BK / 8; ++k8) {       // 8 tf32 = 32 bytes (8 TMEM columns) per instruction
                                    const uint64_t ko = (uint64_t)(k8 * 2);
                                    const uint32_t accum = (kt | k8) ? 1u : 0u;
                                    f3_umma(d_tmem + t * F3_ACC, w_hi + ko, x_hilo + ko, F3_IDESC32, accum);            // hh | hl
                                    f3_umma_ts(d_tmem + t * F3_ACC + 2 * F3_NB, lo_tmem + t * F3_BK + k8 * 8, x_hilo + ko,
                                               F3_IDESC16, accum);                                                        // lh
                                }
                            }
                            umma_commit(bar_raw_empty + rs);         // both slots are free when these MMAs retire
                            umma_commit(bar_lo_empty + ls);
                            if (kt == F3_KT - 1) umma_commit(bar_tfull + as);
                        }
                        __syncwarp();
                    }
                }
    } else if (warp < 6) {
        // ===================== lo parts: w - trunc_tf32(w); W1 lo -> tensor memory, x lo -> behind x hi ==========
        const int pt = threadIdx.x - 64;          // 0..127
        const int q = warp & 3;                   // TMEM lane quarter of this warp
        const int r = q * 32 + lane;              // row of the 128-row tiles this thread owns
        uint32_t it = 0;
        for (int m = blockIdx.x; m < p.P; m += gridDim.x)
            for (int fb = 0; fb < n_fblk; ++fb)
                for (int ps = 0; ps < F3_NPASS; ++ps)
                    for (int kt = 0; kt < F3_KT; ++kt, ++it) {
                        const uint32_t rs = it % F3_R, ruse = it / F3_R, ls = it % F3_L, luse = it / F3_L;
                        if (luse > 0) tc_mbar_wait(bar_lo_empty + ls, (luse - 1) & 1);
                        tc_mbar_wait(bar_raw_full + rs, ruse & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                        unsigned char* slot = raw_mem + (size_t)rs * F3_SLOT;
#pragma unroll
                        for (int t = 0; t < 2; ++t) {
                            // row r of tile t: 128 bytes, 16-byte chunk c stored at c ^ (r & 7)
                            const float4* row = reinterpret_cast<const float4*>(slot + (size_t)(t * 128 + r) * 128);
                            float lo[32];
#pragma unroll
                            for (int c = 0; c < 8; ++c) {
                                const float4 w = row[c ^ (r & 7)];
                                lo[4 * c] = f3_lo(w.x);
                                lo[4 * c + 1] = f3_lo(w.y);
                                lo[4 * c + 2] = f3_lo(w.z);
                                lo[4 * c + 3] = f3_lo(w.w);
                            }
                            f3_tmem_st32(tmem_base + ((uint32_t)(q * 32) << 16) + F3_TM_LO + ls * F3_TM_LSLOT + t * F3_BK, lo);
                        }
                        {   // activations: x lo right behind x hi (128 float4, one per thread)
                            const float4* xs = reinterpret_cast<const float4*>(slot + F3_A_BYTES);
                            float4* xd = reinterpret_cast<float4*>(slot + F3_A_BYTES + F3_X_BYTES);
                            const float4 w = xs[pt];
                            xd[pt] = make_float4(f3_lo(w.x), f3_lo(w.y), f3_lo(w.z), f3_lo(w.w));
                        }
                        asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
                        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic writes -> tensor core reads
                        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                        __syncwarp();
                        if (lane == 0) tc_mbar_arrive(bar_lo_full + ls);
                    }
    } else {
        // ===================== epilogue (warps 6..9) =====================
        const int q = warp & 3;                          // TMEM lane quarter this warp may access
        const int et = (warp - 6) * 32 + lane;           // 0..127
        const int n_out = p.n_act * F3_NB;               // (action, frame) outputs of a frame block
        uint32_t pass = 0;
        for (int m = blockIdx.x; m < p.P; m += gridDim.x) {
            const float* W = p.members + (int64_t)m * p.pitch;
            for (int fb = 0; fb < n_fblk; ++fb) {
                float acc[(F3_MAX_ACT * F3_NB + 127) / 128];
#pragma unroll
                for (int j = 0; j < (F3_MAX_ACT * F3_NB + 127) / 128; ++j) acc[j] = 0.f;
                for (int ps = 0; ps < F3_NPASS; ++ps, ++pass) {
                    const uint32_t as = pass & 1, ause = pass >> 1;
                    tc_mbar_wait(bar_tfull + as, ause & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    asm volatile("bar.sync 1, 128;\n" ::: "memory");         // everyone is done with the previous hs
#pragma unroll
                    for (int t = 0; t < 2; ++t) {
                        uint32_t hh[16], hl[16], lh[16];
                        const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + as * (2 * F3_ACC) + t * F3_ACC;
                        f3_tmem_ld16(ta, hh);
                        f3_tmem_ld16(ta + F3_NB, hl);
                        f3_tmem_ld16(ta + 2 * F3_NB, lh);
                        const int r = t * 128 + q * 32 + lane;                // row inside the pass
                        const float b = __ldg(W + p.f1b_off + ps * F3_ROWS + r);
                        float4* dst = reinterpret_cast<float4*>(hs + r * F3_NB);
                        const int sw = (r >> 1) & 3;
                        float h[16];
#pragma unroll
                        for (int n = 0; n < 16; ++n)           // small terms first, then the bias (like fc1(x) + b)
                            h[n] = fmaxf(((__uint_as_float(lh[n]) + __uint_as_float(hl[n])) + __uint_as_float(hh[n])) + b, 0.f);
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            dst[c ^ sw] = make_float4(h[4 * c], h[4 * c + 1], h[4 * c + 2], h[4 * c + 3]);
                    }
                    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                    __syncwarp();
                    if (lane == 0) tc_mbar_arrive(bar_tempty + as);
                    asm volatile("bar.sync 1, 128;\n" ::: "memory");         // hs of this pass complete
                    // output layer, this pass's 256 hidden units: out[a][n] += sum_r Wout[a][ps*256 + r] * hs[r][n]
#pragma unroll
                    for (int j = 0; j < (F3_MAX_ACT * F3_NB + 127) / 128; ++j) {
                        const int o = et + 128 * j;
                        if (o < n_out) {
                            const int a = o / F3_NB, n = o % F3_NB;
                            const float* wo = W + p.ow_off + a * 512 + ps * F3_ROWS;
                            float s = acc[j];
#pragma unroll 8
                            for (int r = 0; r < F3_ROWS; ++r) {
                                const int sw = (r >> 1) & 3;
                                s = fmaf(__ldg(wo + r), hs[r * F3_NB + (((n >> 2) ^ sw) << 2) + (n & 3)], s);
                            }
                            acc[j] = s;
                        }
                    }
                }
                // logits + first-max argmax of this frame block (the exchange buffer reuses hs)
                asm volatile("bar.sync 1, 128;\n" ::: "memory");
#pragma unroll
                for (int j = 0; j < (F3_MAX_ACT * F3_NB + 127) / 128; ++j) {
                    const int o = et + 128 * j;
                    if (o < n_out) {
                        const int a = o / F3_NB, n = o % F3_NB;
                        const float v = acc[j] + __ldg(W + p.ob_off + a);
                        lgs[a * F3_NB + n] = v;
                        const int frame = fb * F3_NB + n;
                        if (frame < p.B) p.logits[((int64_t)m * p.B + frame) * p.n_act + a] = v;
                    }
                }
                asm volatile("bar.sync 1, 128;\n" ::: "memory");
                if (et < F3_NB && fb * F3_NB + et < p.B && p.actions) {
                    int best = 0;
                    float bv = lgs[et];
                    for (int a = 1; a < p.n_act; ++a) {
                        const float v = lgs[a * F3_NB + et];
                        if (v > bv) { bv = v; best = a; }              // first maximum (Atari/deepqn.py:55-60)
                    }
                    p.actions[(int64_t)m * p.B + fb * F3_NB + et] = best;
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}


// fc1 + output layer + argmax for all members on the tensor cores.
// act3: fp32 [P*B, 3136] (conv3 output, post BN + ReLU, flattened like torch's reshape).
int launch_deepqn_fc_tc(cev_handle* h, const float* members, int64_t pitch, int P, int B, int n_act, int f1w_off,
                        int f1b_off, int ow_off, int ob_off, const float* act3, float* logits, int32_t* actions,
                        cudaStream_t stream) {
    EncodeTiledFn encode = get_encode_fn();
    if (!encode) {
        set_error("deepqn_fc_tc: cuTensorMapEncodeTiled is not available from the driver");
        return CEV_ERR_UNSUPPORTED;
    }
    CEV_REQUIRE(n_act <= F3_MAX_ACT, "deepqn_fc_tc: at most %d actions", F3_MAX_ACT);
    CUtensorMap map_x, map_w;
    {
        // rows past the end of the activation matrix are zero-filled; rows of a neighbouring member only
        // reach accumulator columns of frames >= B, which are never read
        cuuint64_t dims[2] = {(cuuint64_t)F3_K, (cuuint64_t)P * B};
        cuuint64_t strides[1] = {(cuuint64_t)F3_K * 4};
        cuuint32_t box[2] = {F3_BK, F3_NB};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&map_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(act3), dims, strides, box,
                            estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("deepqn_fc_tc: cuTensorMapEncodeTiled(x) failed with %d", (int)r);
            return CEV_ERR_CUDA;
        }
    }
    {
        cuuint64_t dims[3] = {(cuuint64_t)F3_K, 512, (cuuint64_t)P};
        cuuint64_t strides[2] = {(cuuint64_t)F3_K * 4, (cuuint64_t)pitch * 4};
        cuuint32_t box[3] = {F3_BK, F3_ROWS, 1};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = encode(&map_w, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(members + f1w_off), dims,
                            strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            getenv("CEV_K2_L2P128") ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("deepqn_fc_tc: cuTensorMapEncodeTiled(w) failed with %d", (int)r);
            return CEV_ERR_CUDA;
        }
    }
    TcParams p;
    p.members = members;
    p.pitch = pitch;
    p.P = P;
    p.B = B;
    p.n_act = n_act;
    p.f1b_off = f1b_off;
    p.ow_off = ow_off;
    p.ob_off = ob_off;
    p.logits = logits;
    p.actions = actions;
    static bool configured[16] = {};          // a function attribute is per device
    if (h->device < 16 && !configured[h->device]) {
        CEV_CUDA(cudaFuncSetAttribute(deepqn_fc_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)F3_SMEM));
        configured[h->device] = true;
    }
    const int grid = P < h->n_sm ? P : h->n_sm;
    deepqn_fc_tc_kernel<<<grid, F3_THREADS, F3_SMEM, stream>>>(map_x, map_w, p);
    return check_cuda(cudaGetLastError(), "deepqn_fc_tc_kernel");
}

}  // namespace cev
