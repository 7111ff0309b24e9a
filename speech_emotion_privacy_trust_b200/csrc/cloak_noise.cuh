// The cloak's per-element noise and its derivative, shared by the feature cloak (cloak.cu) and the waveform cloak's
// evaluation and per-utterance backward kernels (wave_cloak.cu), so both evaluate one definition of sigma, of
// d sigma / d rho and of mu + sigma * eps.
#pragma once
#include <cuda_runtime.h>

namespace sept {

__device__ __forceinline__ float sigma_of(float rho, float mn, float mx) {
    return __fadd_rn(__fmul_rn((1.0f + tanhf(rho)) / 2.0f, mx - mn), mn);   // operation order of cloak_models.py:43
}

__device__ __forceinline__ float dsigma_of(float rho, float mn, float mx) {
    const float range = mx - mn, th = tanhf(rho);
    return (1.0f - th * th) * 0.5f * range;
}

// product and sum rounded separately, like the reference's two ATen ops (no FMA contraction)
__device__ __forceinline__ float noise_of(float mu, float sigma, float eps) { return __fadd_rn(mu, __fmul_rn(sigma, eps)); }

}  // namespace sept
