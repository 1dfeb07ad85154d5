// K5 device code shared by the isotropic / separable K5 (population_ops.cu) and the guided-search K5
// (es_subspace.cu): the mutation power of a launch and one float4 of a perturbed member row.
#pragma once

#include "common.cuh"

namespace cev {

// sigma of a launch: the by-value argument, or -- when the generation state lives on the device
// (cev_generation_end_f64 adapts it there, SURVEY.md 8f N1) -- the fp64 scalar the caller points at,
// rounded to fp32 exactly like the host's float(sigma).
__device__ __forceinline__ float pick_sigma(float sigma, const double* __restrict__ sigma_dev) {
    return sigma_dev ? (float)__ldg(sigma_dev) : sigma;
}

// CTAs of K5T threads at <= 48 registers: 6 K of the register file, so a perturb CTA of one role can be resident
// next to the rollout kernels' CTAs of another role (two 128-thread member CTAs at 230 registers leave 6.6 K,
// the 448-thread opponent CTA 9 K) and fill their idle issue slots instead of waiting for a free SM.
// Every segment boundary of the row is a multiple of 4 parameters except the end of the row, so a float4 is
// perturbable or not as a whole (the LayerNorm float4s skip the Philox / Box-Muller work altogether).
constexpr int K5T = 128;

// Mutation power of K5: one scalar for the whole row (the isotropic search distribution), or a row of
// per-parameter sigmas laid out like theta (separable NES), read as the float4 of parameters j .. j+3.
struct ScalarSigma {
    float s;
    __device__ __forceinline__ float4 at(int) const { return make_float4(s, s, s, s); }
};
struct RowSigma {
    const float* __restrict__ row;
    __device__ __forceinline__ float4 at(int j) const { return __ldg(reinterpret_cast<const float4*>(row + j)); }
};

// Search direction eps of parameter j + i from its normal z: z itself (isotropic and separable K5), or the guided
// direction fl(fl(A z) + fl(B s_i)) with s_i the subspace term U^T c of that parameter (es_perturb_subspace_kernel).
struct IsoDir {
    __device__ __forceinline__ float operator()(int, float z) const { return z; }
};
struct SubspaceDir {
    float a, b;
    float s[4];
    __device__ __forceinline__ float operator()(int i, float z) const {
        return __fadd_rn(__fmul_rn(a, z), __fmul_rn(b, s[i]));
    }
};

// One float4 (parameters j .. j+3) of K5.  `counter` is the Philox member word: the member id, or the pair id
// q = c >> 1 under mirrored sampling, where the normals of one draw give the row theta + sigma eps (`plus`, the
// even member 2q) and the row theta - sigma eps (`minus`, the odd member 2q+1) with the same rounded product.
// A null row pointer skips that row (a pair cut by the shard boundary); noise rows receive +z / -z.
template <bool MIRROR, class Sigma, class Dir = IsoDir>
__device__ __forceinline__ void es_perturb_float4(
    const float* __restrict__ theta, const FcOffsets& o, int j4, const Sigma& sigma, const PhiloxKeys& keys,
    uint32_t tag, uint32_t gen, uint32_t counter, float* __restrict__ plus, float* __restrict__ minus,
    float* __restrict__ noise_plus, float* __restrict__ noise_minus, const Dir& dir = Dir()) {
    const int j = j4 * 4;
    const float4 pv = __ldg(reinterpret_cast<const float4*>(theta + j));
    float p[4] = {pv.x, pv.y, pv.z, pv.w};
    float m[4] = {pv.x, pv.y, pv.z, pv.w};
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (j < o.total && fc_is_perturbable(o, j)) {
        normal4(keys, tag, gen, counter, (uint32_t)j4, z);
        const float4 sv = sigma.at(j);
        const float s[4] = {sv.x, sv.y, sv.z, sv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (j + i < o.total) {
                const float d = __fmul_rn(s[i], dir(i, z[i]));
                p[i] = __fadd_rn(p[i], d);
                if (MIRROR) m[i] = __fadd_rn(m[i], -d);
            } else { z[i] = 0.f; p[i] = 0.f; m[i] = 0.f; }
        }
    } else if (j >= o.total) {
        p[0] = p[1] = p[2] = p[3] = 0.f;
        m[0] = m[1] = m[2] = m[3] = 0.f;
    }
    if (!MIRROR || plus) __stcs(reinterpret_cast<float4*>(plus + j), make_float4(p[0], p[1], p[2], p[3]));
    if (MIRROR && minus) __stcs(reinterpret_cast<float4*>(minus + j), make_float4(m[0], m[1], m[2], m[3]));
    if (noise_plus)
        *reinterpret_cast<float4*>(noise_plus + j) = make_float4(z[0], z[1], z[2], z[3]);
    if (MIRROR && noise_minus)
        *reinterpret_cast<float4*>(noise_minus + j) = make_float4(-z[0], -z[1], -z[2], -z[3]);
}

}  // namespace cev
