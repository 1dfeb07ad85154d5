// Co-GA safe mutations through output gradients (SM-G-SUM, Lehman, Chen, Clune & Stanley, GECCO 2018): the
// per-parameter scale rows of the elites (cev_ga_safe_scale_f32) and K3 with a scale row (cev_ga_repopulate_safe_f32).
// A translation unit of its own: ptxas allocates the registers of the kernels of one module together, so apart from
// them every existing kernel keeps its SASS.
//
// For a parent row W and the 32 probe observations x_t of the novelty search, with y_k(x_t) the logits:
//   G_kj = sum_t dy_k(x_t) / dW_j,  s_j = sqrt(sum_k G_kj^2),  c_j = 1 if s_j == 0, else 1 / max(s_j, floor).
// The chain of one parent: a forward over the 32 probes, then the 5 x 32 backward rows (one per (logit, probe)).
// Five launches, each over (tiles x) parents, so a few parents still spread over many SMs:
//   1. layer 1 + LayerNorm 1                       grid E          -> a1, xhat1, rstd1
//   2. layer 2 (fc2 rows in 32-unit tiles)         grid 8 x E      -> h2
//   3. LayerNorm 2, logits, the output layer's and LayerNorm 2's backward; scales of fc2.b, ln2, out   grid E -> dz2
//   4. fc2 in 32-column tiles: G(fc2.W) = dz2^T a1 and da1 = dz2 W2   grid 16 x E   -> fc2.W scales, da1
//   5. LayerNorm 1's backward; scales of fc1, ln1 and the zero padding   grid E
// Intermediates live in the handle's workspace.  Every sum runs in a fixed order (no atomics), and nothing depends
// on E or on which CTA computes a parent, so a parent's row is the same in any launch.  FP32 FFMA throughout.
#include <algorithm>

#include "common.cuh"
#include "es_perturb.cuh"

namespace cev {

constexpr int SM_P = CEV_NOVELTY_PROBES;      // probe observations (the batch of the sensitivity)
constexpr int SM_ROWS = NACT * SM_P;          // backward rows per parent
constexpr int SM_T = 256;
constexpr int SM_UT = 32;                     // fc2 rows (layer-2 units) per CTA of the layer-2 forward
constexpr int SM_CT = 32;                     // fc2 columns (layer-1 units) per CTA of the fc2 backward
constexpr int SM_W2LD = H1 + 1;               // padded row stride of an fc2 row tile in shared memory
static_assert(SM_T == H2 && 2 * SM_T == H1, "thread i owns layer-2 unit i");

// workspace of one parent, in floats
constexpr int64_t WS_A1 = 0;                               // [32][512] layer-1 activations
constexpr int64_t WS_X1 = WS_A1 + SM_P * H1;               // [32][512] normalised layer-1 pre-activations
constexpr int64_t WS_R1 = WS_X1 + SM_P * H1;               // [32] 1 / sqrt(var + eps) of LayerNorm 1 (64 reserved)
constexpr int64_t WS_H2 = WS_R1 + 64;                      // [32][256] layer-2 pre-activations
constexpr int64_t WS_DZ2 = WS_H2 + SM_P * H2;              // [5][32][256] d y_k / d (fc2 output)
constexpr int64_t WS_DA1 = WS_DZ2 + SM_ROWS * H2;          // [5][32][512] d y_k / d (layer-1 activations)
constexpr int64_t WS_PER = WS_DA1 + SM_ROWS * H1;
static_assert(WS_PER % 4 == 0, "parents' workspaces stay 16-byte aligned");

__device__ __forceinline__ float sm_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;                                            // the same bits in every lane (each step is commutative)
}

// c of an entry from s^2 = sum_k G_k^2; a non-finite one sets the status word
__device__ __forceinline__ float sm_scale(float s2, float floor_, int32_t* status) {
    if (!isfinite(s2) && status) atomicOr(status, CEV_STATUS_NONFINITE);
    const float s = sqrtf(s2);
    return s == 0.f ? 1.f : __frcp_rn(fmaxf(s, floor_));
}

// LayerNorm (biased variance, eps 1e-5) of row x[0 .. N) by one warp, the forward kernels' arithmetic: writes the
// normalised row xhat, the activation relu(xhat * g + b) (a NaN stays NaN) and returns 1 / sqrt(var + eps).
template <int N>
__device__ __forceinline__ float sm_layer_norm_row(const float* x, const float* __restrict__ g,
                                                   const float* __restrict__ b, float* xhat, float* act, int lane) {
    constexpr int V = N / 32;
    float v[V];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        v[i] = x[lane + 32 * i];
        s += v[i];
    }
    const float mean = sm_warp_sum(s) * (1.0f / N);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        v[i] -= mean;
        q = fmaf(v[i], v[i], q);
    }
    const float var = sm_warp_sum(q) * (1.0f / N);
    const float rstd = 1.0f / sqrtf(var + LN_EPS);
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const float xh = v[i] * rstd;
        const float y = fmaf(xh, __ldg(g + lane + 32 * i), __ldg(b + lane + 32 * i));
        xhat[lane + 32 * i] = xh;
        act[lane + 32 * i] = y < 0.f ? 0.f : y;
    }
    return rstd;
}

// LayerNorm backward of one row by one warp: dh = rstd (dxh - mean(dxh) - xhat mean(dxh xhat)), dxh = dy g
template <int N>
__device__ __forceinline__ void sm_layer_norm_back_row(const float* dxh, const float* xhat, float rstd, float* dh,
                                                       int lane) {
    constexpr int V = N / 32;
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
        s1 += dxh[lane + 32 * i];
        s2 = fmaf(dxh[lane + 32 * i], xhat[lane + 32 * i], s2);
    }
    const float m1 = sm_warp_sum(s1) * (1.0f / N);
    const float m2 = sm_warp_sum(s2) * (1.0f / N);
#pragma unroll
    for (int i = 0; i < V; ++i) {
        const int u = lane + 32 * i;
        dh[u] = rstd * (dxh[u] - m1 - xhat[u] * m2);
    }
}

// ---- 1. layer 1 + LayerNorm 1 (grid E, 256 threads) ----------------------------------------------------------
template <int IN>
__global__ void __launch_bounds__(SM_T) sm_fwd1_kernel(const float* __restrict__ rows, int64_t pitch,
                                                      const float* __restrict__ obs, float* __restrict__ ws) {
    __shared__ float so[SM_P * IN];
    __shared__ float h1[SM_P * H1 / 4];                  // a quarter of the probes at a time
    constexpr FcOffsets o = fc_offsets(IN);
    const float* W = rows + (int64_t)blockIdx.x * pitch;
    float* w = ws + (int64_t)blockIdx.x * WS_PER;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < SM_P * IN; i += SM_T) so[i] = obs[i];
    float wr[2][IN], br[2];
#pragma unroll
    for (int uu = 0; uu < 2; ++uu) {
#pragma unroll
        for (int i = 0; i < IN; ++i) wr[uu][i] = __ldg(W + o.fc1w + (tid + uu * SM_T) * IN + i);
        br[uu] = __ldg(W + o.fc1b + tid + uu * SM_T);
    }
    for (int t0 = 0; t0 < SM_P; t0 += SM_P / 4) {
        __syncthreads();
        for (int tt = 0; tt < SM_P / 4; ++tt) {
#pragma unroll
            for (int uu = 0; uu < 2; ++uu) {
                float acc = 0.f;
#pragma unroll
                for (int i = 0; i < IN; ++i) acc = fmaf(so[(t0 + tt) * IN + i], wr[uu][i], acc);
                h1[tt * H1 + tid + uu * SM_T] = acc + br[uu];
            }
        }
        __syncthreads();
        const int t = t0 + warp;                         // 8 warps, 8 probes per quarter
        const float r = sm_layer_norm_row<H1>(h1 + warp * H1, W + o.ln1g, W + o.ln1b, w + WS_X1 + t * H1,
                                              w + WS_A1 + t * H1, lane);
        if (lane == 0) w[WS_R1 + t] = r;
    }
}

// ---- 2. layer 2: h2 = a1 W2^T + b2 for 32 fc2 rows (grid 8 x E, 256 threads) -----------------------------------
__global__ void __launch_bounds__(SM_T) sm_fwd2_kernel(const float* __restrict__ rows, int64_t pitch, int in_dim,
                                                      float* __restrict__ ws) {
    extern __shared__ float4 sm_smem[];
    float* a1 = reinterpret_cast<float*>(sm_smem);       // [32][512]
    float* w2 = a1 + SM_P * H1;                          // [32][SM_W2LD]
    const FcOffsets o = fc_offsets(in_dim);
    const int i0 = blockIdx.x * SM_UT;
    const float* W = rows + (int64_t)blockIdx.y * pitch;
    float* w = ws + (int64_t)blockIdx.y * WS_PER;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int q = tid; q < SM_P * H1 / 4; q += SM_T)
        reinterpret_cast<float4*>(a1)[q] = reinterpret_cast<const float4*>(w + WS_A1)[q];
    for (int q = tid; q < SM_UT * H1; q += SM_T) {
        const int u = q / H1, j = q - u * H1;
        w2[u * SM_W2LD + j] = __ldg(W + o.fc2w + (int64_t)(i0 + u) * H1 + j);
    }
    __syncthreads();
    // thread: unit i0 + lane, probes 4 warp .. 4 warp + 3
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    const float* wr = w2 + lane * SM_W2LD;
    const float* ar = a1 + (4 * warp) * H1;
    for (int j = 0; j < H1; ++j) {
        const float wv = wr[j];
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) acc[tt] = fmaf(ar[tt * H1 + j], wv, acc[tt]);
    }
    const float b = __ldg(W + o.fc2b + i0 + lane);
#pragma unroll
    for (int tt = 0; tt < 4; ++tt) w[WS_H2 + (4 * warp + tt) * H2 + i0 + lane] = acc[tt] + b;
}

// ---- 3. LayerNorm 2, logits, backward to dz2; scales of fc2.b, ln2, out (grid E, 256 threads) ------------------
__global__ void __launch_bounds__(SM_T) sm_mid_kernel(const float* __restrict__ rows, int64_t pitch, int in_dim,
                                                     float floor_, float* __restrict__ scale, int64_t scale_pitch,
                                                     float* __restrict__ ws, int32_t* __restrict__ status) {
    extern __shared__ float4 sm_smem[];
    float* xh = reinterpret_cast<float*>(sm_smem);       // [32][256] normalised h2
    float* a2 = xh + SM_P * H2;                          // [32][256] layer-2 activations
    float* dxh = a2 + SM_P * H2;                         // [32][256] dy2 * g2 of the current logit
    float* dz = dxh + SM_P * H2;                         // [32][256] dz2 of the current logit
    __shared__ float rstd[SM_P];
    const FcOffsets o = fc_offsets(in_dim);
    const float* W = rows + (int64_t)blockIdx.x * pitch;
    float* w = ws + (int64_t)blockIdx.x * WS_PER;
    float* S = scale + (int64_t)blockIdx.x * scale_pitch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int t = warp; t < SM_P; t += SM_T / 32) {
        const float r = sm_layer_norm_row<H2>(w + WS_H2 + t * H2, W + o.ln2g, W + o.ln2b, xh + t * H2, a2 + t * H2,
                                              lane);
        if (lane == 0) rstd[t] = r;
    }
    __syncthreads();
    // logits: a non-finite one sets the status word
    for (int t = warp; t < SM_P; t += SM_T / 32) {
        bool fin = true;
#pragma unroll
        for (int k = 0; k < NACT; ++k) {
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < H2 / 32; ++q) s = fmaf(a2[t * H2 + lane + 32 * q], __ldg(W + o.outw + k * H2 + lane + 32 * q), s);
            fin = fin && isfinite(sm_warp_sum(s) + __ldg(W + o.outb + k));
        }
        if (!fin && lane == 0 && status) atomicOr(status, CEV_STATUS_NONFINITE);
    }
    // output layer: dy_k / d out.W[k'][i] = [k == k'] a2_t[i], dy_k / d out.b[k'] = [k == k']
    const int i = tid;
    float ga = 0.f;
    for (int t = 0; t < SM_P; ++t) ga += a2[t * H2 + i];
    const float g2 = __ldg(W + o.ln2g + i);
    float s_b2 = 0.f, s_g2 = 0.f, s_be2 = 0.f;
    for (int k = 0; k < NACT; ++k) {
        const float wo = __ldg(W + o.outw + k * H2 + i);
        float gg = 0.f, gb = 0.f;
        for (int t = 0; t < SM_P; ++t) {                  // dy2 = [a2 > 0] out.W[k][i]
            const float dy = a2[t * H2 + i] > 0.f ? wo : 0.f;
            dxh[t * H2 + i] = dy * g2;
            gg = fmaf(dy, xh[t * H2 + i], gg);
            gb += dy;
        }
        s_g2 = fmaf(gg, gg, s_g2);
        s_be2 = fmaf(gb, gb, s_be2);
        __syncthreads();
        for (int t = warp; t < SM_P; t += SM_T / 32)
            sm_layer_norm_back_row<H2>(dxh + t * H2, xh + t * H2, rstd[t], dz + t * H2, lane);
        __syncthreads();
        float gz = 0.f;
        for (int t = 0; t < SM_P; ++t) {
            const float v = dz[t * H2 + i];
            w[WS_DZ2 + (k * SM_P + t) * H2 + i] = v;
            gz += v;
        }
        s_b2 = fmaf(gz, gz, s_b2);
        __syncthreads();                                  // dxh / dz are rewritten for the next logit
    }
    S[o.fc2b + i] = sm_scale(s_b2, floor_, status);
    S[o.ln2g + i] = sm_scale(s_g2, floor_, status);
    S[o.ln2b + i] = sm_scale(s_be2, floor_, status);
    const float c_out = sm_scale(fmaf(ga, ga, 0.f), floor_, status);
#pragma unroll
    for (int k = 0; k < NACT; ++k) S[o.outw + k * H2 + i] = c_out;
    if (i < NACT) S[o.outb + i] = sm_scale((float)(SM_P * SM_P), floor_, status);
}

// ---- 4. fc2 in 32-column tiles: G(fc2.W)[i][j] = sum_t dz2[t][i] a1[t][j] and da1[t][j] = sum_i dz2[t][i] W2[i][j]
//      (grid 16 x E, 256 threads: lane = column j0 + lane; warp w: units w + 8 r, probes 4 w .. 4 w + 3) ----------
__global__ void __launch_bounds__(SM_T) sm_w2_kernel(const float* __restrict__ rows, int64_t pitch, int in_dim,
                                                    float floor_, float* __restrict__ scale, int64_t scale_pitch,
                                                    float* __restrict__ ws, int32_t* __restrict__ status) {
    extern __shared__ float4 sm_smem[];
    float* dzs = reinterpret_cast<float*>(sm_smem);      // [32][256] dz2 of the current logit
    float* w2 = dzs + SM_P * H2;                         // [256][32] the column tile of W2
    const FcOffsets o = fc_offsets(in_dim);
    const int j0 = blockIdx.x * SM_CT;
    const float* W = rows + (int64_t)blockIdx.y * pitch;
    float* w = ws + (int64_t)blockIdx.y * WS_PER;
    float* S = scale + (int64_t)blockIdx.y * scale_pitch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int u = warp; u < H2; u += SM_T / 32) w2[u * SM_CT + lane] = __ldg(W + o.fc2w + (int64_t)u * H1 + j0 + lane);
    float a1c[SM_P];
#pragma unroll
    for (int t = 0; t < SM_P; ++t) a1c[t] = w[WS_A1 + t * H1 + j0 + lane];
    float s2[H2 / 8];
#pragma unroll
    for (int r = 0; r < H2 / 8; ++r) s2[r] = 0.f;
    for (int k = 0; k < NACT; ++k) {
        __syncthreads();
        for (int q = tid; q < SM_P * H2 / 4; q += SM_T)
            reinterpret_cast<float4*>(dzs)[q] = reinterpret_cast<const float4*>(w + WS_DZ2 + k * SM_P * H2)[q];
        __syncthreads();
#pragma unroll
        for (int r = 0; r < H2 / 8; ++r) {
            const int i = warp + 8 * r;
            float g = 0.f;
#pragma unroll
            for (int t = 0; t < SM_P; ++t) g = fmaf(dzs[t * H2 + i], a1c[t], g);
            s2[r] = fmaf(g, g, s2[r]);
        }
        float acc[4] = {0.f, 0.f, 0.f, 0.f};
        const float* dr = dzs + (4 * warp) * H2;
#pragma unroll 4
        for (int i = 0; i < H2; ++i) {
            const float wv = w2[i * SM_CT + lane];
#pragma unroll
            for (int tt = 0; tt < 4; ++tt) acc[tt] = fmaf(dr[tt * H2 + i], wv, acc[tt]);
        }
#pragma unroll
        for (int tt = 0; tt < 4; ++tt) w[WS_DA1 + (k * SM_P + 4 * warp + tt) * H1 + j0 + lane] = acc[tt];
    }
#pragma unroll
    for (int r = 0; r < H2 / 8; ++r)
        S[o.fc2w + (int64_t)(warp + 8 * r) * H1 + j0 + lane] = sm_scale(s2[r], floor_, status);
}

// ---- 5. LayerNorm 1's backward; scales of fc1, ln1 and the padding (grid E, 512 threads) ------------------------
template <int IN>
__global__ void __launch_bounds__(2 * SM_T) sm_back1_kernel(const float* __restrict__ rows, int64_t pitch,
                                                           const float* __restrict__ obs, float floor_,
                                                           float* __restrict__ scale, int64_t scale_pitch,
                                                           const float* __restrict__ ws, int32_t* __restrict__ status) {
    extern __shared__ float4 sm_smem[];
    float* dxh = reinterpret_cast<float*>(sm_smem);      // [32][512] dy1 * g1 of the current logit
    float* dz = dxh + SM_P * H1;                         // [32][512] dz1 of the current logit
    __shared__ float so[SM_P * IN];
    constexpr FcOffsets o = fc_offsets(IN);
    const float* W = rows + (int64_t)blockIdx.x * pitch;
    const float* w = ws + (int64_t)blockIdx.x * WS_PER;
    float* S = scale + (int64_t)blockIdx.x * scale_pitch;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int q = tid; q < SM_P * IN; q += 2 * SM_T) so[q] = obs[q];
    const int j = tid;                                   // layer-1 unit
    const float g1 = __ldg(W + o.ln1g + j);
    float s_g1 = 0.f, s_be1 = 0.f, s_b1 = 0.f, s_w1[IN];
#pragma unroll
    for (int i = 0; i < IN; ++i) s_w1[i] = 0.f;
    for (int k = 0; k < NACT; ++k) {
        const float* da = w + WS_DA1 + k * SM_P * H1;
        float gg = 0.f, gb = 0.f;
        for (int t = 0; t < SM_P; ++t) {                  // dy1 = [a1 > 0] da1
            const float dy = w[WS_A1 + t * H1 + j] > 0.f ? da[t * H1 + j] : 0.f;
            dxh[t * H1 + j] = dy * g1;
            gg = fmaf(dy, w[WS_X1 + t * H1 + j], gg);
            gb += dy;
        }
        s_g1 = fmaf(gg, gg, s_g1);
        s_be1 = fmaf(gb, gb, s_be1);
        __syncthreads();
        for (int t = warp; t < SM_P; t += 2 * SM_T / 32)
            sm_layer_norm_back_row<H1>(dxh + t * H1, w + WS_X1 + t * H1, w[WS_R1 + t], dz + t * H1, lane);
        __syncthreads();
        float gz = 0.f, gw[IN];
#pragma unroll
        for (int i = 0; i < IN; ++i) gw[i] = 0.f;
        for (int t = 0; t < SM_P; ++t) {
            const float v = dz[t * H1 + j];
            gz += v;
#pragma unroll
            for (int i = 0; i < IN; ++i) gw[i] = fmaf(v, so[t * IN + i], gw[i]);
        }
        s_b1 = fmaf(gz, gz, s_b1);
#pragma unroll
        for (int i = 0; i < IN; ++i) s_w1[i] = fmaf(gw[i], gw[i], s_w1[i]);
        __syncthreads();                                  // dxh / dz are rewritten for the next logit
    }
#pragma unroll
    for (int i = 0; i < IN; ++i) S[o.fc1w + j * IN + i] = sm_scale(s_w1[i], floor_, status);
    S[o.fc1b + j] = sm_scale(s_b1, floor_, status);
    S[o.ln1g + j] = sm_scale(s_g1, floor_, status);
    S[o.ln1b + j] = sm_scale(s_be1, floor_, status);
    for (int64_t q = o.total + tid; q < scale_pitch; q += 2 * SM_T) S[q] = 0.f;
}

// ---- K3 with a scale row: child c >= 1 = fl(p + fl(fl(sigma z) c)), c from the elite p was copied from --------
// ga_repopulate_kernel (population_ops.cu) with the scale rows: the same parents, crossover mask and normals.  The
// body is restated here rather than shared through a template: instantiating K3's body from a header changes
// ptxas's instruction order for the existing kernel, whose SASS stays as it is.
constexpr int SK_T = 256;
__global__ void __launch_bounds__(SK_T) ga_repopulate_safe_kernel(
    const float* __restrict__ elites, const float* __restrict__ scale, int E, int D, int64_t pitch, float sigma_arg,
    const double* __restrict__ sigma_dev, const PhiloxKeys keys, uint32_t tag, uint32_t gen, int64_t row0,
    float xrate, uint32_t xtag, float* __restrict__ out, float* __restrict__ noise_out) {
    const float sigma = pick_sigma(sigma_arg, sigma_dev);
    const int64_t r = blockIdx.x;
    const int64_t c = row0 + r;                       // global member id
    const int j4 = blockIdx.y * SK_T + threadIdx.x;
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
    const float4 sv = __ldg(reinterpret_cast<const float4*>(scale + parent * pitch + (int64_t)j4 * 4));
    float s[4] = {sv.x, sv.y, sv.z, sv.w};
    if (mate >= 0) {
        const float4 qv = *reinterpret_cast<const float4*>(elites + mate * pitch + (int64_t)j4 * 4);
        const float4 tv = __ldg(reinterpret_cast<const float4*>(scale + mate * pitch + (int64_t)j4 * 4));
        const U4 x = philox4x32_10(U4{(uint32_t)j4, (uint32_t)c, gen, xtag}, keys);
        if (!(x.x & 1u)) { p[0] = qv.x; s[0] = tv.x; }
        if (!(x.y & 1u)) { p[1] = qv.y; s[1] = tv.y; }
        if (!(x.z & 1u)) { p[2] = qv.z; s[2] = tv.z; }
        if (!(x.w & 1u)) { p[3] = qv.w; s[3] = tv.w; }
    }
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (c != 0) {
        normal4(keys, tag, gen, (uint32_t)c, (uint32_t)j4, z);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int j = j4 * 4 + i;
            if (j < D) p[i] = __fadd_rn(p[i], __fmul_rn(__fmul_rn(sigma, z[i]), s[i]));
            else { p[i] = 0.f; z[i] = 0.f; }
        }
    }
    *reinterpret_cast<float4*>(out + r * pitch + (int64_t)j4 * 4) = make_float4(p[0], p[1], p[2], p[3]);
    if (noise_out)
        *reinterpret_cast<float4*>(noise_out + r * pitch + (int64_t)j4 * 4) = make_float4(z[0], z[1], z[2], z[3]);
}

}  // namespace cev

using namespace cev;

static bool sm_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// the dynamic shared memory of the kernels above, set once per device (a function attribute is per device)
static int sm_configure(int device) {
    static bool done[16] = {};
    if (device < 16 && done[device]) return CEV_OK;
    const int fwd2 = (int)((SM_P * H1 + SM_UT * SM_W2LD) * sizeof(float));
    CEV_CUDA(cudaFuncSetAttribute(sm_fwd2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, fwd2));
    CEV_CUDA(cudaFuncSetAttribute(sm_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(4 * SM_P * H2 * sizeof(float))));
    CEV_CUDA(cudaFuncSetAttribute(sm_w2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)((SM_P * H2 + H2 * SM_CT) * sizeof(float))));
    CEV_CUDA(cudaFuncSetAttribute(sm_back1_kernel<IN_ADV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(2 * SM_P * H1 * sizeof(float))));
    CEV_CUDA(cudaFuncSetAttribute(sm_back1_kernel<IN_GOOD>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)(2 * SM_P * H1 * sizeof(float))));
    if (device < 16) done[device] = true;
    return CEV_OK;
}

template <int IN>
static int sm_launch(cev_handle* h, const float* rows, int64_t pitch, int E, const float* obs, float floor_,
                     float* scale, int64_t scale_pitch, int32_t* status, cudaStream_t st) {
    float* ws = static_cast<float*>(h->workspace);
    sm_fwd1_kernel<IN><<<E, SM_T, 0, st>>>(rows, pitch, obs, ws);
    CEV_CUDA(cudaGetLastError());
    sm_fwd2_kernel<<<dim3(H2 / SM_UT, E), SM_T, (SM_P * H1 + SM_UT * SM_W2LD) * sizeof(float), st>>>(rows, pitch, IN,
                                                                                                    ws);
    CEV_CUDA(cudaGetLastError());
    sm_mid_kernel<<<E, SM_T, 4 * SM_P * H2 * sizeof(float), st>>>(rows, pitch, IN, floor_, scale, scale_pitch, ws,
                                                                 status);
    CEV_CUDA(cudaGetLastError());
    sm_w2_kernel<<<dim3(H1 / SM_CT, E), SM_T, (SM_P * H2 + H2 * SM_CT) * sizeof(float), st>>>(
        rows, pitch, IN, floor_, scale, scale_pitch, ws, status);
    CEV_CUDA(cudaGetLastError());
    sm_back1_kernel<IN><<<E, 2 * SM_T, 2 * SM_P * H1 * sizeof(float), st>>>(rows, pitch, obs, floor_, scale,
                                                                             scale_pitch, ws, status);
    return check_cuda(cudaGetLastError(), "sm_back1_kernel");
}

extern "C" {

int cev_ga_safe_scale_f32(cev_handle* h, const float* rows, int64_t pitch, int in_dim, int E, const float* probe_obs,
                          float floor_, float* scale, int64_t scale_pitch, int32_t* status, cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "ga_safe_scale: null handle");
    CEV_REQUIRE(in_dim == IN_ADV || in_dim == IN_GOOD, "ga_safe_scale: in_dim must be 8 or 10");
    CEV_REQUIRE(E >= 0 && E <= 65535, "ga_safe_scale: need 0 <= E <= 65535");
    CEV_REQUIRE(isfinite(floor_) && floor_ > 0.f, "ga_safe_scale: floor must be finite and > 0");
    if (E == 0) return CEV_OK;
    CEV_REQUIRE(rows && probe_obs && scale, "ga_safe_scale: null pointer");
    const int D = fc_offsets(in_dim).total;
    CEV_REQUIRE(pitch >= D && pitch % 4 == 0 && scale_pitch >= D && scale_pitch % 4 == 0,
                "ga_safe_scale: row pitches must be multiples of 4 floats >= %d", D);
    CEV_REQUIRE(sm_aligned16(rows) && sm_aligned16(scale), "ga_safe_scale: rows must be 16-byte aligned");
    CEV_GUARD(h);
    const size_t need = (size_t)E * WS_PER * sizeof(float);
    if (h->workspace_bytes < need) {
        if (h->workspace) cudaFree(h->workspace);
        h->workspace = nullptr;
        h->workspace_bytes = 0;
        CEV_CUDA(cudaMalloc(&h->workspace, need));
        h->workspace_bytes = need;
    }
    const int rc = sm_configure(h->device);
    if (rc != CEV_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (in_dim == IN_ADV) return sm_launch<IN_ADV>(h, rows, pitch, E, probe_obs, floor_, scale, scale_pitch, status, st);
    return sm_launch<IN_GOOD>(h, rows, pitch, E, probe_obs, floor_, scale, scale_pitch, status, st);
}

int cev_ga_repopulate_safe_f32(cev_handle* h, const float* elites, const float* scale, int E, int D, int64_t pitch,
                               float sigma, const double* sigma_dev, float crossover_rate, uint64_t seed, int role,
                               uint32_t gen, int64_t row0, int64_t n_rows, float* out, float* noise_out,
                               cev_stream stream) {
    CEV_REQUIRE(h != nullptr, "ga_repopulate_safe: null handle");
    if (n_rows == 0) return CEV_OK;                   // an empty shard contributes nothing
    CEV_REQUIRE(elites && scale && out, "ga_repopulate_safe: null pointer");
    CEV_REQUIRE(E >= 1 && D >= 1 && pitch >= D && pitch % 4 == 0, "ga_repopulate_safe: bad E/D/pitch");
    CEV_REQUIRE(crossover_rate >= 0.f && crossover_rate <= 1.f,
                "ga_repopulate_safe: crossover_rate must be in [0, 1]");
    CEV_REQUIRE(sm_aligned16(elites) && sm_aligned16(scale) && sm_aligned16(out) && sm_aligned16(noise_out),
                "ga_repopulate_safe: 16B alignment");
    CEV_REQUIRE(row0 >= 0 && n_rows >= 0 && row0 + n_rows <= 0xFFFFFFFFll, "ga_repopulate_safe: bad row range");
    CEV_GUARD(h);
    const uint32_t k0 = (uint32_t)(seed & 0xFFFFFFFFull), k1 = (uint32_t)(seed >> 32);
    dim3 grid((unsigned)n_rows, (unsigned)((pitch / 4 + SK_T - 1) / SK_T));
    ga_repopulate_safe_kernel<<<grid, SK_T, 0, (cudaStream_t)stream>>>(
        elites, scale, E, D, pitch, sigma, sigma_dev, philox_keys(k0, k1), noise_tag(CEV_KIND_GA, role), gen, row0,
        crossover_rate, noise_tag(CEV_KIND_XOVER, role), out, noise_out);
    return check_cuda(cudaGetLastError(), "ga_repopulate_safe_kernel");
}

}  // extern "C"
