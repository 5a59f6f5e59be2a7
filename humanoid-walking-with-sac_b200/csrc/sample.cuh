// Tanh-Gaussian sampling arithmetic shared by the T_SAMPLE / T_SAMPLE_BWD tasks and the forward / select_action kernels (extras.cu).
#pragma once
#include "common.cuh"

namespace sacb {

// ---- Philox4x32-10 (Salmon et al. 2011) for production-mode eps draws --------------------------------------
__device__ __forceinline__ void philox4x32(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
        c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
__device__ __forceinline__ float philox_normal(uint64_t seed, uint32_t stream, uint32_t step, uint32_t row, uint32_t col) {
    uint32_t c[4] = {row, col, step, stream};
    philox4x32(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const float u1 = ((float)(c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(c[1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
    return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// tanh-Gaussian sample of one action component: networks_model1.py:83-96 == networks_model2.py:104-117
struct SampleElem { float action, logp, y, std, in_range; };
__device__ __forceinline__ SampleElem sample_elem(float mean, float ls_raw, float eps, float scale, float bias) {
    SampleElem o;
    const float ls = fminf(fmaxf(ls_raw, kLogStdMin), kLogStdMax);     // torch.clamp(log_std, -20, 2)
    o.in_range = (ls_raw >= kLogStdMin && ls_raw <= kLogStdMax) ? 1.f : 0.f;
    o.std = expf(ls);
    const float x = mean + eps * o.std;                                  // Normal.rsample
    o.y = tanhf(x);
    o.action = o.y * scale + bias;
    const float var = o.std * o.std;
    const float d = x - mean;
    float lp = -(d * d) / (2.f * var) - logf(o.std) - kLogSqrt2Pi;      // Normal.log_prob
    lp -= logf(scale * (1.f - o.y * o.y) + kSquashEps);
    o.logp = lp;
    return o;
}

}  // namespace sacb
