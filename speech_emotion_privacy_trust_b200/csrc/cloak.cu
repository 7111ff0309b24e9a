// Cloak noise layer + gradient reversal, fused (sm_100a).
//
//   cloak_fwd_kernel   out[b,i] = x[b,i]*mask[i] + locs[i] + sigma(rhos[i]) * eps[i]*mask[i]
//                      sigma = (1 + tanh rho)/2 * (max - min) + min; eps either supplied by the caller or drawn on
//                      the device (Philox4x32-10 + Box-Muller, std 0.1), one (W,F) sample broadcast over the batch.
//                      Replaces cloak_noise.scales/sample_noise/forward (model/cloak_models.py:41-58): ~10 ATen
//                      launches + a CPU RNG + an H2D copy become one launch.
//   cloak_bwd_kernel   g = g_a - lambda * g_b (the second upstream gradient arrives through a gradient-reversal
//                      layer, model/reversal_gradient.py:19-23); dlocs = sum_b g; drhos = dlocs * eps*mask * dsigma/drho
//                      (+ the -scale_lambda * log(mean sigma) regulariser's gradient when asked); dx = g*mask.
//                      Deterministic: batch slices write partial sums, the last CTA of a column adds them in order.
//   grl_bwd_kernel     dx = -lambda * g (stand-alone GradientReversal backward).
//
// HBM-bound, zero reuse: float4 accesses, grid sized so that every SM has work at B = 32..64.
#include <cuda_runtime.h>
#include <cstdint>

#include "cloak.h"
#include "cloak_noise.cuh"
#include "philox.cuh"

namespace sept {

__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

constexpr int kCloakThreads = 128;

__device__ __forceinline__ float4 cloak_noise4(const CloakFwdParams& p, float4 mu, float4 rho, float4 e, float4 m) {
    if (p.mask) { e.x *= m.x; e.y *= m.y; e.z *= m.z; e.w *= m.w; }
    float4 nz;
    nz.x = noise_of(mu.x, sigma_of(rho.x, p.min_scale, p.max_scale), e.x);
    nz.y = noise_of(mu.y, sigma_of(rho.y, p.min_scale, p.max_scale), e.y);
    nz.z = noise_of(mu.z, sigma_of(rho.z, p.min_scale, p.max_scale), e.z);
    nz.w = noise_of(mu.w, sigma_of(rho.w, p.min_scale, p.max_scale), e.w);
    return nz;
}

__global__ void __launch_bounds__(kCloakThreads) cloak_fwd_kernel(const CloakFwdParams p) {
    const int i4 = blockIdx.x * kCloakThreads + threadIdx.x;
    if (i4 * 4 >= p.wf) return;
    const int i = i4 * 4;
    const uint64_t quads = (uint64_t)((p.wf + 3) / 4);
    const uint64_t off = p.draw_dev ? p.offset + *p.draw_dev * quads : p.offset;
    const float4 mu = ld4(p.locs + i), rho = ld4(p.rhos + i);
    const float4 m = p.mask ? ld4(p.mask + i) : make_float4(1.f, 1.f, 1.f, 1.f);
    float4 nz = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!p.per_sample) {
        const float4 e = p.eps ? ld4(p.eps + i) : normal4(p.seed, off, (uint32_t)i4, p.eps_std);
        if (p.eps_out && blockIdx.y == 0) st4(p.eps_out + i, e);
        nz = cloak_noise4(p, mu, rho, e, m);
        if (p.noise_out && blockIdx.y == 0) st4(p.noise_out + i, nz);
    }
    if (!p.per_sample) {
        // shared eps: four batch rows per trip, all loads issued before the first store (the kernel is latency bound:
        // 13 MB per launch is ~2 us of HBM time)
        const int step = gridDim.y;
        for (int b = blockIdx.y; b < p.batch; b += 4 * step) {
            float4 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (b + j * step < p.batch) v[j] = __ldcs(reinterpret_cast<const float4*>(p.x + (size_t)(b + j * step) * p.wf + i));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (b + j * step >= p.batch) break;
                float4 t = v[j];
                if (p.mask) { t.x = __fmul_rn(t.x, m.x); t.y = __fmul_rn(t.y, m.y); t.z = __fmul_rn(t.z, m.z); t.w = __fmul_rn(t.w, m.w); }
                t.x = __fadd_rn(t.x, nz.x); t.y = __fadd_rn(t.y, nz.y); t.z = __fadd_rn(t.z, nz.z); t.w = __fadd_rn(t.w, nz.w);
                st4(p.out + (size_t)(b + j * step) * p.wf + i, t);
            }
        }
        return;
    }
    for (int b = blockIdx.y; b < p.batch; b += gridDim.y) {
        const size_t o = (size_t)b * p.wf + i;
        const float4 e = p.eps ? ld4(p.eps + o) : normal4(p.seed, off + (uint64_t)b * quads, (uint32_t)i4, p.eps_std);
        if (p.eps_out) st4(p.eps_out + o, e);
        nz = cloak_noise4(p, mu, rho, e, m);
        float4 v = ld4(p.x + o);
        if (p.mask) { v.x = __fmul_rn(v.x, m.x); v.y = __fmul_rn(v.y, m.y); v.z = __fmul_rn(v.z, m.z); v.w = __fmul_rn(v.w, m.w); }
        v.x = __fadd_rn(v.x, nz.x); v.y = __fadd_rn(v.y, nz.y); v.z = __fadd_rn(v.z, nz.z); v.w = __fadd_rn(v.w, nz.w);
        st4(p.out + o, v);
    }
}

__global__ void __launch_bounds__(kCloakThreads) cloak_bwd_kernel(const CloakBwdParams p) {
    const int i4 = blockIdx.x * kCloakThreads + threadIdx.x;
    const int i = i4 * 4;
    const bool live = i < p.wf;
    float4 m = make_float4(1.f, 1.f, 1.f, 1.f);
    if (live && p.mask) m = ld4(p.mask + i);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    if (live) {
        const int step = gridDim.y;
        for (int b = blockIdx.y; b < p.batch; b += 4 * step) {     // four batch rows (eight loads) in flight per thread
            float4 ga[4], gb[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const bool on = b + j * step < p.batch;
                const size_t o = (size_t)(b + j * step) * p.wf + i;
                ga[j] = on ? __ldcs(reinterpret_cast<const float4*>(p.g_a + o)) : make_float4(0.f, 0.f, 0.f, 0.f);
                gb[j] = (on && p.g_b) ? __ldcs(reinterpret_cast<const float4*>(p.g_b + o)) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                if (b + j * step >= p.batch) break;
                float4 g = ga[j];
                const float4 h = gb[j];
                g.x -= p.lambda * h.x; g.y -= p.lambda * h.y; g.z -= p.lambda * h.z; g.w -= p.lambda * h.w;
                s.x += g.x; s.y += g.y; s.z += g.z; s.w += g.w;
                if (p.dx) st4(p.dx + (size_t)(b + j * step) * p.wf + i, make_float4(g.x * m.x, g.y * m.y, g.z * m.z, g.w * m.w));
            }
        }
        st4(p.partial + (size_t)blockIdx.y * p.wf + i, s);
    }
    // ---- last CTA of this column folds the slices in order ----------------------------------------------------
    __shared__ int is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned done = atomicAdd(p.counters + blockIdx.x, 1u);
        is_last = (done == gridDim.y - 1);
        if (is_last) p.counters[blockIdx.x] = 0u;                // ready for the next call
    }
    __syncthreads();
    if (!is_last || !live) return;
    __threadfence();
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (unsigned sl = 0; sl < gridDim.y; ++sl) {
        const float4 v = __ldcg(reinterpret_cast<const float4*>(p.partial + (size_t)sl * p.wf + i));
        t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    st4(p.dlocs + i, t);
    if (p.drhos) {
        const float4 rho = ld4(p.rhos + i), e = ld4(p.eps + i);
        const float ds[4] = {dsigma_of(rho.x, p.min_scale, p.max_scale), dsigma_of(rho.y, p.min_scale, p.max_scale),
                             dsigma_of(rho.z, p.min_scale, p.max_scale), dsigma_of(rho.w, p.min_scale, p.max_scale)};
        const float em[4] = {e.x * m.x, e.y * m.y, e.z * m.z, e.w * m.w};
        const float tt[4] = {t.x, t.y, t.z, t.w};
        float r[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            // reg_coef = -scale_lambda / (wf * mean sigma): gradient of -scale_lambda * log(mean(sigma)) wrt sigma_i
            r[c] = (tt[c] * em[c] + p.reg_coef) * ds[c];
        }
        st4(p.drhos + i, make_float4(r[0], r[1], r[2], r[3]));
    }
}

__global__ void __launch_bounds__(256) grl_bwd_kernel(const float* __restrict__ g, float neg_lambda, size_t n,
                                                       float* __restrict__ dx) {
    const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
    for (size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
        if (i + 4 <= n) {
            const float4 v = ld4(g + i);
            st4(dx + i, make_float4(neg_lambda * v.x, neg_lambda * v.y, neg_lambda * v.z, neg_lambda * v.w));
        } else {
            for (size_t j = i; j < n; ++j) dx[j] = neg_lambda * g[j];
        }
    }
}

__global__ void counter_add_kernel(uint64_t* c, uint64_t inc) { *c += inc; }

cudaError_t launch_counter_add(uint64_t* counter, uint64_t inc, cudaStream_t stream) {
    counter_add_kernel<<<1, 1, 0, stream>>>(counter, inc);
    return cudaGetLastError();
}

int cloak_slices(int batch) { return batch < kCloakSlices ? (batch > 0 ? batch : 1) : kCloakSlices; }

cudaError_t launch_cloak_fwd(const CloakFwdParams& p, cudaStream_t stream) {
    const int blocks = (p.wf / 4 + kCloakThreads - 1) / kCloakThreads;
    dim3 grid(blocks, cloak_slices(p.batch));
    cloak_fwd_kernel<<<grid, kCloakThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_cloak_bwd(const CloakBwdParams& p, cudaStream_t stream) {
    const int blocks = (p.wf / 4 + kCloakThreads - 1) / kCloakThreads;
    dim3 grid(blocks, cloak_slices(p.batch));
    cloak_bwd_kernel<<<grid, kCloakThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_grl_bwd(const float* g, float lambda, size_t n, float* dx, cudaStream_t stream) {
    if (n == 0) return cudaSuccess;
    size_t blocks = (n / 4 + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    if (blocks == 0) blocks = 1;
    grl_bwd_kernel<<<(unsigned)blocks, 256, 0, stream>>>(g, -lambda, n, dx);
    return cudaGetLastError();
}

}  // namespace sept
