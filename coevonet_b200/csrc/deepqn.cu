// K2 -- grouped per-member DeepQN forward (Atari/deepqn.py:39-48).
//
// One CTA per population member; the member's frames are processed layer by layer
// so every weight tensor is read from HBM exactly once per member:
//   x/255 -> conv 8x8/4 (C->32) -> BN -> ReLU -> conv 4x4/2 (32->64) -> BN -> ReLU
//         -> conv 3x3/1 (64->64) -> BN -> ReLU -> flatten(3136) -> FC 512 -> ReLU -> FC A
// The "virtual batch norm" layers are train-mode BatchNorm2d at batch 1
// (SURVEY.md Appendix C #12): statistics per frame over H x W, biased variance.
//
// Round-1 state: FP32 CUDA-core arithmetic (parity first: logits within 1e-5 of
// the reference's fp32 forward).  Conv weights are staged transposed in shared
// memory ([k][cout], so lanes over output channels are conflict-free) and reused
// for all frames of the member; the 6.4 MB fc1 matrix -- 95 % of a member's bytes --
// is streamed once with 128-bit loads and reused across the member's frames, which
// makes the kernel HBM-bound on weight bytes at small frames-per-member (roofline
// in DESIGN.md section 6).  The tcgen05/TMA implicit-GEMM version of the four
// contractions is the round-2 item for this kernel.
#include <stdlib.h>
#include <string.h>

#include "deepqn_common.cuh"

namespace cev {

constexpr int DQ_T = 256;
constexpr int DQ_FB = 12;                 // frames per fc pass (12 x (3136 + 512) floats = 175 KB of shared memory)

// stage conv weights W[cout][k] (global, k contiguous) as Wt[k][cout] in shared memory.
// (A padded-tile transposition that removes the shared-memory store conflicts was measured
// slower -- two block barriers per 32-k tile -- so the direct form stays.)
template <int COUT>
__device__ __forceinline__ void stage_weights_transposed(const float* __restrict__ w, int K, float* wt,
                                                         float* /*tile, unused*/) {
    for (int i = threadIdx.x; i < COUT * K; i += DQ_T) {
        const int c = i / K, k = i - c * K;
        wt[k * COUT + c] = __ldg(w + i);
    }
}

// Direct convolution + bias for one frame held in shared memory.
// Thread = (channel quad cq, position slot ps); 4 channels x 4 positions per step.
template <int CIN, int COUT, int KS, int STRIDE, int HIN, int HOUT, typename InT>
__device__ __forceinline__ void conv_frame(const InT* __restrict__ in_s, const float* __restrict__ lut,
                                           const float* __restrict__ wt, const float* __restrict__ bias,
                                           float* __restrict__ out_s) {
    constexpr int NQ = COUT / 4;                 // channel quads
    constexpr int NPS = DQ_T / NQ;               // position slots
    constexpr int NPOS = HOUT * HOUT;
    constexpr int K = CIN * KS * KS;
    const int cq = threadIdx.x % NQ, ps = threadIdx.x / NQ;
    const float4 b4 = *reinterpret_cast<const float4*>(bias + 4 * cq);
    for (int p0 = ps * 4; p0 < NPOS; p0 += NPS * 4) {
        int base[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int p = min(p0 + j, NPOS - 1);
            base[j] = (p / HOUT) * STRIDE * HIN + (p % HOUT) * STRIDE;
        }
        float acc[4][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[j][0] = 0.f; acc[j][1] = 0.f; acc[j][2] = 0.f; acc[j][3] = 0.f; }
        int k = 0;
        for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
            for (int ky = 0; ky < KS; ++ky) {
#pragma unroll
                for (int kx = 0; kx < KS; ++kx, ++k) {
                    const float4 w = *reinterpret_cast<const float4*>(wt + k * COUT + 4 * cq);
                    const int off = ci * HIN * HIN + ky * HIN + kx;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float x;
                        if constexpr (sizeof(InT) == 1) x = lut[in_s[base[j] + off]];
                        else x = (float)in_s[base[j] + off];
                        acc[j][0] = fmaf(w.x, x, acc[j][0]);
                        acc[j][1] = fmaf(w.y, x, acc[j][1]);
                        acc[j][2] = fmaf(w.z, x, acc[j][2]);
                        acc[j][3] = fmaf(w.w, x, acc[j][3]);
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int p = p0 + j;
            if (p < NPOS) {
                out_s[(4 * cq + 0) * NPOS + p] = acc[j][0] + b4.x;
                out_s[(4 * cq + 1) * NPOS + p] = acc[j][1] + b4.y;
                out_s[(4 * cq + 2) * NPOS + p] = acc[j][2] + b4.z;
                out_s[(4 * cq + 3) * NPOS + p] = acc[j][3] + b4.w;
            }
        }
    }
    (void)K;
}

// train-mode BatchNorm (per frame, per channel over NPOS positions) + ReLU, in place,
// then copy to global.  One warp per channel (round robin).
template <int COUT, int NPOS>
__device__ __forceinline__ void bn_relu_store(float* __restrict__ out_s, const float* __restrict__ gamma,
                                              const float* __restrict__ beta, float* __restrict__ dst) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int c = warp; c < COUT; c += DQ_T / 32) {
        float* row = out_s + c * NPOS;
        const float x0 = row[0];      // sums of deviations from it: a constant channel normalises to exactly beta
        float s = 0.f;
        for (int p = lane; p < NPOS; p += 32) s += row[p] - x0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = x0 + s * (1.0f / NPOS);
        float q = 0.f;
        for (int p = lane; p < NPOS; p += 32) {
            const float d = row[p] - mean;
            q = fmaf(d, d, q);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = 1.0f / sqrtf(q * (1.0f / NPOS) + BN_EPS);
        const float g = __ldg(gamma + c), b = __ldg(beta + c);
        for (int p = lane; p < NPOS; p += 32) {
            const float v = fmaxf(fmaf((row[p] - mean) * rstd, g, b), 0.f);
            dst[c * NPOS + p] = v;
        }
    }
}

struct DqnParams {
    const float* members;
    int64_t pitch;
    const uint8_t* frames;
    int P, B, c_in, n_act;
    float* act1;       // [P][B][32*400]
    float* act2;       // [P][B][64*81]
    float* act3;       // [P][B][3136]
    float* logits;
    int32_t* actions;
    int skip_fc;       // 1: the tensor-core stage (deepqn_tc.cu) computes fc1 / output / argmax
};

template <int CIN>
__global__ void __launch_bounds__(DQ_T, 1) deepqn_forward_kernel(const DqnParams p) {
    extern __shared__ __align__(16) unsigned char dq_smem[];
    const DqnOffsets o = dqn_offsets(CIN, p.n_act);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int m = blockIdx.x; m < p.P; m += gridDim.x) {
        const float* W = p.members + (int64_t)m * p.pitch;
        float* a1 = p.act1 + (int64_t)m * p.B * 12800;
        float* a2 = p.act2 + (int64_t)m * p.B * 5184;
        float* a3 = p.act3 + (int64_t)m * p.B * 3136;
        // ---------------- conv1: u8 frame [CIN][84][84] -> [32][20][20] -------------
        {
            float* wt = reinterpret_cast<float*>(dq_smem);                    // [CIN*64][32]
            float* out_s = wt + CIN * 64 * 32;                                // [32][400]
            float* lut = out_s + 12800;                                       // [256]
            uint8_t* in_s = reinterpret_cast<uint8_t*>(lut + 256);            // [CIN][84][84]
            float* tile = reinterpret_cast<float*>(in_s + CIN * 7056);        // [32][33]
            __syncthreads();
            stage_weights_transposed<32>(W + o.c1w, CIN * 64, wt, tile);
            for (int i = threadIdx.x; i < 256; i += DQ_T) lut[i] = __fdiv_rn((float)i, 255.0f);
            for (int f = 0; f < p.B; ++f) {
                const uint8_t* fr = p.frames + ((int64_t)m * p.B + f) * CIN * 7056;
                __syncthreads();
                for (int i = threadIdx.x; i < CIN * 7056 / 16; i += DQ_T)
                    reinterpret_cast<uint4*>(in_s)[i] = __ldg(reinterpret_cast<const uint4*>(fr) + i);
                __syncthreads();
                conv_frame<CIN, 32, 8, 4, 84, 20, uint8_t>(in_s, lut, wt, W + o.c1b, out_s);
                __syncthreads();
                bn_relu_store<32, 400>(out_s, W + o.bn1g, W + o.bn1b, a1 + (int64_t)f * 12800);
            }
        }
        // ---------------- conv2: [32][20][20] -> [64][9][9] ---------------------------
        {
            float* wt = reinterpret_cast<float*>(dq_smem);                    // [512][64]
            float* in_s = wt + 512 * 64;                                      // [32][400]
            float* out_s = in_s + 12800;                                      // [64][81]
            float* tile = out_s + 5184;                                       // [64][33]
            __syncthreads();
            stage_weights_transposed<64>(W + o.c2w, 512, wt, tile);
            for (int f = 0; f < p.B; ++f) {
                __syncthreads();
                for (int i = threadIdx.x; i < 12800 / 4; i += DQ_T)
                    reinterpret_cast<float4*>(in_s)[i] = reinterpret_cast<const float4*>(a1 + (int64_t)f * 12800)[i];
                __syncthreads();
                conv_frame<32, 64, 4, 2, 20, 9, float>(in_s, nullptr, wt, W + o.c2b, out_s);
                __syncthreads();
                bn_relu_store<64, 81>(out_s, W + o.bn2g, W + o.bn2b, a2 + (int64_t)f * 5184);
            }
        }
        // ---------------- conv3: [64][9][9] -> [64][7][7] ------------------------------
        {
            float* wt = reinterpret_cast<float*>(dq_smem);                    // [576][64]
            float* in_s = wt + 576 * 64;                                      // [64][81]
            float* out_s = in_s + 5184;                                       // [64][49]
            float* tile = out_s + 3136;                                       // [64][33]
            __syncthreads();
            stage_weights_transposed<64>(W + o.c3w, 576, wt, tile);
            for (int f = 0; f < p.B; ++f) {
                __syncthreads();
                for (int i = threadIdx.x; i < 5184 / 4; i += DQ_T)
                    reinterpret_cast<float4*>(in_s)[i] = reinterpret_cast<const float4*>(a2 + (int64_t)f * 5184)[i];
                __syncthreads();
                conv_frame<64, 64, 3, 1, 9, 7, float>(in_s, nullptr, wt, W + o.c3b, out_s);
                __syncthreads();
                bn_relu_store<64, 49>(out_s, W + o.bn3g, W + o.bn3b, a3 + (int64_t)f * 3136);
            }
        }
        // ---------------- fc1 (3136 -> 512) + ReLU, out (512 -> A), argmax ---------------
        for (int f0 = 0; f0 < p.B && !p.skip_fc; f0 += DQ_FB) {
            const int nb = min(DQ_FB, p.B - f0);
            float* x_s = reinterpret_cast<float*>(dq_smem);                   // [DQ_FB][3136]
            float* h_s = x_s + DQ_FB * 3136;                                  // [DQ_FB][512]
            __syncthreads();
            for (int i = threadIdx.x; i < nb * 3136 / 4; i += DQ_T)
                reinterpret_cast<float4*>(x_s)[i] = reinterpret_cast<const float4*>(a3 + (int64_t)f0 * 3136)[i];
            for (int i = nb * 3136 + threadIdx.x; i < DQ_FB * 3136; i += DQ_T) x_s[i] = 0.f;
            __syncthreads();
            for (int n = warp; n < 512; n += DQ_T / 32) {
                const float4* wr = reinterpret_cast<const float4*>(W + o.f1w + (int64_t)n * 3136);
                float4 w[25];
#pragma unroll
                for (int i = 0; i < 25; ++i) {
                    const int q = lane + 32 * i;                              // float4 index, 784 per row
                    w[i] = q < 784 ? __ldg(wr + q) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                const float bias = __ldg(W + o.f1b + n);
                for (int b = 0; b < DQ_FB; ++b) {
                    if (b >= nb) break;
                    const float4* xr = reinterpret_cast<const float4*>(x_s + b * 3136);
                    float acc = 0.f;
#pragma unroll
                    for (int i = 0; i < 25; ++i) {
                        const int q = lane + 32 * i;
                        if (q < 784) {
                            const float4 x = xr[q];
                            acc = fmaf(w[i].x, x.x, acc);
                            acc = fmaf(w[i].y, x.y, acc);
                            acc = fmaf(w[i].z, x.z, acc);
                            acc = fmaf(w[i].w, x.w, acc);
                        }
                    }
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                    if (lane == 0) h_s[b * 512 + n] = fmaxf(acc + bias, 0.f);
                }
            }
            __syncthreads();
            // output layer: one warp per (frame, action)
            for (int job = warp; job < nb * p.n_act; job += DQ_T / 32) {
                const int b = job / p.n_act, a = job % p.n_act;
                const float* wr = W + o.ow + a * 512;
                float acc = 0.f;
#pragma unroll
                for (int i = 0; i < 16; ++i) acc = fmaf(__ldg(wr + lane + 32 * i), h_s[b * 512 + lane + 32 * i], acc);
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
                if (lane == 0) p.logits[((int64_t)m * p.B + f0 + b) * p.n_act + a] = acc + __ldg(W + o.ob + a);
            }
            __syncthreads();
            if (p.actions) {
                for (int b = threadIdx.x; b < nb; b += DQ_T) {
                    const float* lg = p.logits + ((int64_t)m * p.B + f0 + b) * p.n_act;
                    int best = 0;
                    float bv = lg[0];
                    for (int a = 1; a < p.n_act; ++a)
                        if (lg[a] > bv) { bv = lg[a]; best = a; }      // first maximum (Atari/deepqn.py:55-60)
                    p.actions[(int64_t)m * p.B + f0 + b] = best;
                }
            }
        }
    }
}

static size_t dqn_smem_bytes(int c_in) {
    const size_t conv1 = (size_t)(c_in * 64 * 32 + 12800 + 256 + 32 * 33) * 4 + (size_t)c_in * 7056;
    const size_t conv2 = (size_t)(512 * 64 + 12800 + 5184 + 64 * 33) * 4;
    const size_t conv3 = (size_t)(576 * 64 + 5184 + 3136 + 64 * 33) * 4;
    const size_t fc = (size_t)(DQ_FB * 3136 + DQ_FB * 512) * 4;
    size_t m = conv1 > conv2 ? conv1 : conv2;
    m = m > conv3 ? m : conv3;
    return m > fc ? m : fc;
}

}  // namespace cev

using namespace cev;

extern "C" int cev_deepqn_forward(cev_handle* h, const float* members, int P, int64_t pitch,
                                  const uint8_t* frames, int B, int c_in, int n_actions, float* logits,
                                  int32_t* actions, cev_stream stream) {
    CEV_REQUIRE(h && members && frames && logits, "deepqn_forward: null pointer");
    CEV_REQUIRE(c_in == 4 || c_in == 6, "deepqn_forward: c_in must be 4 (synthetic frames) or 6 (reference wrapper chain)");
    CEV_REQUIRE(n_actions >= 1 && n_actions <= 32 && P >= 0 && B >= 1, "deepqn_forward: bad P/B/n_actions");
    const DqnOffsets o = dqn_offsets(c_in, n_actions);
    CEV_REQUIRE(pitch >= o.total && pitch % 4 == 0, "deepqn_forward: pitch too small / not a multiple of 4");
    CEV_REQUIRE((reinterpret_cast<uintptr_t>(members) & 15u) == 0 && (reinterpret_cast<uintptr_t>(frames) & 15u) == 0,
                "deepqn_forward: rows and frames must be 16B aligned");
    if (P == 0) return CEV_OK;
    CEV_GUARD(h);
    // activation scratch (stays in L2 between the layer phases of a member)
    const size_t per = (size_t)P * B;
    const size_t need = per * (12800 + 5184 + 3136 + 3136) * sizeof(float);
    if (h->workspace_bytes < need) {
        if (h->workspace) CEV_CUDA(cudaFree(h->workspace));
        h->workspace = nullptr;
        h->workspace_bytes = 0;
        CEV_CUDA(cudaMalloc(&h->workspace, need));
        h->workspace_bytes = need;
    }
    DqnParams p;
    p.members = members;
    p.pitch = pitch;
    p.frames = frames;
    p.P = P;
    p.B = B;
    p.c_in = c_in;
    p.n_act = n_actions;
    p.act1 = static_cast<float*>(h->workspace);
    p.act2 = p.act1 + per * 12800;
    p.act3 = p.act2 + per * 5184;
    float* y3 = p.act3 + per * 3136;          // conv3's pre-BatchNorm output (tensor-core conv path)
    p.logits = logits;
    p.actions = actions;
    // fully-connected stage: tcgen05 (3xTF32, fp32-level accuracy; default) or the fp32 CUDA-core loop
    // (COEVONET_DQN_FC=fp32); convolution stack: tcgen05 implicit GEMM (3xTF32, default with the tensor-core fc
    // stage) or the fp32 CUDA-core kernel (COEVONET_DQN_CONV=fp32, and always with COEVONET_DQN_FC=fp32).
    // Both stages meet the same 2e-5 tolerance against the reference's fp32 forward.
    const char* fc_env = getenv("COEVONET_DQN_FC");
    const bool use_tc = !(fc_env && strcmp(fc_env, "fp32") == 0);
    const char* conv_env = getenv("COEVONET_DQN_CONV");
    const bool conv_tc = use_tc && !(conv_env && strcmp(conv_env, "fp32") == 0);
    p.skip_fc = use_tc ? 1 : 0;
    if (conv_tc) {
        int rc = launch_deepqn_conv_tc(h, members, pitch, P, B, c_in, n_actions, frames, p.act1, p.act2, y3, p.act3,
                                       (cudaStream_t)stream);
        if (rc) return rc;
    } else {
        const size_t smem = dqn_smem_bytes(c_in);
        const int grid = P < h->n_sm ? P : h->n_sm;
        if (c_in == 4) {
            CEV_CUDA(cudaFuncSetAttribute(deepqn_forward_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem));
            deepqn_forward_kernel<4><<<grid, DQ_T, smem, (cudaStream_t)stream>>>(p);
        } else {
            CEV_CUDA(cudaFuncSetAttribute(deepqn_forward_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem));
            deepqn_forward_kernel<6><<<grid, DQ_T, smem, (cudaStream_t)stream>>>(p);
        }
        CEV_CUDA(cudaGetLastError());
    }
    if (use_tc)
        return launch_deepqn_fc_tc(h, members, pitch, P, B, n_actions, o.f1w, o.f1b, o.ow, o.ob, p.act3, logits,
                                   actions, (cudaStream_t)stream);
    return CEV_OK;
}
