// Band-limited sinc resampling of a ragged batch (sm_100a), e.g. 44.1 kHz -> 16 kHz ahead of framing.
//
// Replaces torchaudio.transforms.Resample(sample_rate, 16000) as called for the MSP-Improv corpus
// (feature_extraction/audio_feature_extraction.py:139-141 -> torchaudio/functional/functional.py
// _get_sinc_resample_kernel / _apply_sinc_resample_kernel): Hann-windowed sinc, lowpass_filter_width 6, rolloff 0.99,
// evaluated as `up` polyphase FIR rows applied with stride `orig`.  torchaudio convolves every row over its full
// 2*width + orig taps; outside |t| < lowpass_filter_width the window is cos^2(pi/2) ~ 1e-33, so each row is stored and
// applied on its ~2*width + 2 tap support only (the dropped taps are below fp32 resolution of the sum by > 25 orders).
//
// One thread per output sample: y[m*up + j] = sum_k w[j][k] * x[m*orig + k - width].  Neighbouring outputs read
// overlapping input windows, which L1 serves; the 160 x 36 weight table stays L1 resident.  HBM-bound by a wide margin
// is not reached: 34 FMAs per 6.8 bytes of traffic put it at the L1/FMA balance point.
#include <cuda_runtime.h>
#include <cstdint>

#include "resample.h"
#include "resample_shape.h"
#include "vec.cuh"

namespace sept {

constexpr int kResampleThreads = 256;

__global__ void __launch_bounds__(kResampleThreads) resample_kernel(const ResampleParams p) {
    __shared__ int u_first;
    const long long g0 = (long long)blockIdx.x * kResampleThreads;
    if (threadIdx.x == 0) {
        int lo = 0, hi = p.n_utts - 1;                         // utterance of the block's first output sample
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (p.out_off[mid + 1] > g0) hi = mid; else lo = mid + 1;
        }
        u_first = lo;
    }
    __syncthreads();
    const long long g = g0 + threadIdx.x;
    if (g >= p.total_out) return;
    int u = u_first;
    while (g >= p.out_off[u + 1]) ++u;                         // a block rarely spans more than two utterances
    const long long o = g - p.out_off[u];
    const long long m = o / p.up;
    const int j = (int)(o - m * p.up);
    const long long base = p.in_off[u];
    const long long n_in = p.in_off[u + 1] - base;
    const int k0 = p.k_lo[j];
    const float* w = p.w + (long long)j * p.taps;
    const long long i0 = m * p.orig + k0 - p.width;            // input index of the first stored tap
    const float* x = p.in + base;
    float acc = 0.f;
    if (i0 >= 0 && i0 + p.taps <= n_in) {
#pragma unroll 4
        for (int k = 0; k < p.taps; ++k) acc = fmaf(__ldg(w + k), __ldg(x + i0 + k), acc);
    } else {
        for (int k = 0; k < p.taps; ++k) {
            const long long i = i0 + k;
            if (i >= 0 && i < n_in) acc = fmaf(__ldg(w + k), __ldg(x + i), acc);   // zero padding outside the utterance
        }
    }
    p.out[g] = acc;
}

// ---- tiled kernel ---------------------------------------------------------------------------------------------------
// The one-thread-per-sample kernel above issues two loads per FMA and runs at the L1 request rate (2.4 ms per
// audio-hour at 44.1 -> 16 kHz, eight times the log-mel kernel).  Here a CTA owns kOutRows * up consecutive output
// samples; it stages the input span they need in shared memory (zero padded outside the utterance, which is exactly
// torchaudio's padding) next to the grouped weight table, and a thread computes a 4 x 4 tile -- four consecutive phases
// j of four consecutive rows m (output sample m * up + j) -- walking once over the group's TG-tap window: one 16-byte
// weight load and four input loads feed sixteen FMAs.  Accumulation runs over ascending taps like the kernel above.
// A CTA is two independent halves of kTileThreads threads that share the weight table and each walk their own chunk
// range with their own stage and their own named barrier: a third more resident warps for the same shared memory.
__device__ __forceinline__ void half_barrier(int half) { asm volatile("bar.sync %0, %1;" ::"r"(half + 1), "n"(kTileThreads) : "memory"); }

template <int TG>                                      // TG > 0: p.tg == TG, the tap loop is unrolled; 0: any tap count
__global__ void __launch_bounds__(2 * kTileThreads) resample_tiled_kernel(const ResampleParams p) {
    const int half = threadIdx.x / kTileThreads, tid = threadIdx.x % kTileThreads;
    extern __shared__ __align__(16) unsigned char rs_smem[];
    float4* wt = reinterpret_cast<float4*>(rs_smem);                                  // [n_groups][tg]
    int* base = reinterpret_cast<int*>(wt + p.n_groups * p.tg);                       // [n_groups]
    const TileGeom geo = resample_tile_geom(p.orig, p.n_groups, p.tg, p.base_min, p.base_max);
    float* stage = reinterpret_cast<float*>(base + ((p.n_groups + 3) & ~3)) + half * geo.stage_floats;
    __shared__ int u_first_sh[2];
    int& u_first = u_first_sh[half];
    const long long per_cta = (long long)geo.rows_per_cta * p.up;
    for (int i = threadIdx.x; i < p.n_groups * p.tg; i += 2 * kTileThreads) wt[i] = reinterpret_cast<const float4*>(p.tile_wt)[i];
    for (int i = threadIdx.x; i < p.n_groups; i += 2 * kTileThreads) base[i] = p.tile_base[i];
    __syncthreads();
    // persistent CTAs: the weight table is fetched once, then the CTA walks over its CONTIGUOUS range of chunks of
    // rows_per_cta * up samples -- the utterance of a chunk's first sample is found by one binary search per CTA and a
    // short forward walk per chunk (a search per chunk, ten dependent global loads by one thread, cost more than the
    // chunk's arithmetic)
    const long long n_chunks = (p.total_out + per_cta - 1) / per_cta;
    const long long n_workers = 2LL * gridDim.x, worker = 2LL * blockIdx.x + half;
    const long long c_begin = n_chunks * worker / n_workers, c_end = n_chunks * (worker + 1) / n_workers;
    if (tid == 0) {
        const long long g_first = c_begin * per_cta;
        int lo = 0, hi = p.n_utts - 1;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (p.out_off[mid + 1] > g_first) hi = mid; else lo = mid + 1;
        }
        u_first = lo;
    }
    for (long long chunk = c_begin; chunk < c_end; ++chunk) {
    const long long g0 = chunk * per_cta;
    long long g1 = g0 + per_cta;
    if (g1 > p.total_out) g1 = p.total_out;
    half_barrier(half);                                                                  // u_first is set / the previous chunk is done
    if (tid == 0) {
        int u = u_first;
        while (u < p.n_utts - 1 && p.out_off[u + 1] <= g0) ++u;
        u_first = u;
    }
    half_barrier(half);
    for (int u = u_first; u < p.n_utts && p.out_off[u] < g1; ++u) {
        const long long oo = p.out_off[u], n_out = p.out_off[u + 1] - oo;
        if (n_out <= 0) continue;
        const long long o_lo = g0 > oo ? g0 - oo : 0, o_hi = (g1 - oo < n_out) ? g1 - oo : n_out;   // this CTA's samples of u
        if (o_hi <= o_lo) continue;
        const long long m_lo = o_lo / p.up, m_hi = (o_hi - 1) / p.up;
        const int n_mg = (int)((m_hi - m_lo) / 4 + 1);
        const long long in0 = p.in_off[u], n_in = p.in_off[u + 1] - in0;
        const long long s0 = m_lo * p.orig + p.base_min - p.width;                    // input index of stage[0]
        const int n_stage = (4 * n_mg - 1) * p.orig + (p.base_max - p.base_min) + p.tg;
        half_barrier(half);                                                              // the previous segment's reads are done
        // the span is staged from the 16-byte boundary below its first sample (`shift` floats earlier), so that an
        // interior span moves with 16-byte loads; stage[shift + i] is input sample s0 + i
        const float* src0 = p.in + in0 + s0;
        const int shift = (int)((reinterpret_cast<uintptr_t>(src0) >> 2) & 3);
        const float* src = src0 - shift;
        const int n_fill = n_stage + shift;
        if (s0 - shift >= 0 && s0 - shift + ((n_fill + 3) & ~3) <= n_in) {            // interior: no bounds tests, 16-byte loads
            // asynchronous 16-byte copies (LDGSTS): the whole span is in flight at once and costs no registers -- one trip
            // to memory per stage instead of one per unrolled group of loads; the fill latency is what this kernel waits for
            const float4* src4 = reinterpret_cast<const float4*>(src);
            const unsigned dst = (unsigned)__cvta_generic_to_shared(stage);
            const int n4 = (n_fill + 3) / 4;
            for (int i = tid; i < n4; i += kTileThreads)
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (unsigned)i), "l"(src4 + i) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        } else {
            for (int i = tid; i < n_fill; i += kTileThreads) {
                const long long idx = s0 - shift + i;
                stage[i] = (idx >= 0 && idx < n_in) ? __ldg(src + i) : 0.f;
            }
        }
        half_barrier(half);
        for (int tile = tid; tile < n_mg * p.n_groups; tile += kTileThreads) {
            const int g = tile % p.n_groups, mg = tile / p.n_groups;
            const float4* w = wt + g * p.tg;
            const float* x0 = stage + shift + (4 * mg) * p.orig + (base[g] - p.base_min);
            const float* x1 = x0 + p.orig;
            const float* x2 = x1 + p.orig;
            const float* x3 = x2 + p.orig;
            // packed FP32: a pk2 carries two neighbouring phases; the input sample is the broadcast operand of the FFMA2
            struct alignas(16) w4 { pk2 lo2, hi2; };
            const w4* wp = reinterpret_cast<const w4*>(w);
            pk2 acc2[4][2];
#pragma unroll
            for (int r = 0; r < 4; ++r) { acc2[r][0] = splat(0.f); acc2[r][1] = splat(0.f); }
            auto tap = [&](int i) {
                const w4 wi = wp[i];
                const float xv[4] = {x0[i], x1[i], x2[i], x3[i]};
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const pk2 xs = splat(xv[r]);
                    acc2[r][0] = fma2(wi.lo2, xs, acc2[r][0]);
                    acc2[r][1] = fma2(wi.hi2, xs, acc2[r][1]);
                }
            };
            if constexpr (TG > 0) {                    // known tap count: straight-line code, the loads run ahead of their FMAs
#pragma unroll
                for (int i = 0; i < TG; ++i) tap(i);
            } else {
#pragma unroll 4
                for (int i = 0; i < p.tg; ++i) tap(i);
            }
            float acc[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                acc[r][0] = lo(acc2[r][0]); acc[r][1] = hi(acc2[r][0]);
                acc[r][2] = lo(acc2[r][1]); acc[r][3] = hi(acc2[r][1]);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const long long o = (m_lo + 4 * mg + r) * p.up + 4 * g;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (4 * g + c < p.up && o + c >= o_lo && o + c < o_hi) p.out[oo + o + c] = acc[r][c];
            }
        }
    }
    }
}

// 16-bit PCM -> float in [-1, 1): x / 32768, what torchaudio.load(normalize=True) does on the host before the reference's
// callables see the audio (audio_feature_extraction.py:182).  Lets a bulk job ship half the bytes over PCIe.
__global__ void __launch_bounds__(256) pcm16_to_f32_kernel(const short* __restrict__ in, long long n, float* __restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = (float)in[i] * (1.0f / 32768.0f);
}

cudaError_t launch_pcm16_to_f32(const short* in, long long n, float* out, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    long long blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    pcm16_to_f32_kernel<<<(unsigned)blocks, 256, 0, stream>>>(in, n, out);
    return cudaGetLastError();
}

cudaError_t launch_resample(const ResampleParams& p, cudaStream_t stream) {
    if (p.total_out <= 0) return cudaSuccess;
    const ResampleShape s = resample_shape(p.tile_wt != nullptr, p.orig, p.n_groups, p.tg, p.base_min, p.base_max);
    if (s.kernel != kResampleSimple) {
        const long long per_cta = (long long)s.geo.rows_per_cta * p.up;
        long long blocks = (p.total_out + per_cta - 1) / per_cta;
        const long long resident = 148LL * s.ctas_per_sm;         // CTAs of two independent halves
        if (blocks > resident) blocks = resident;                  // persistent: the weight table is loaded once per CTA
        auto kern = s.kernel == kResampleTiledFast ? resample_tiled_kernel<kTileTapsFast> : resample_tiled_kernel<0>;
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem);
        if (e != cudaSuccess) return e;
        kern<<<(unsigned)blocks, 2 * kTileThreads, s.smem, stream>>>(p);
        return cudaGetLastError();
    }
    const long long blocks = (p.total_out + kResampleThreads - 1) / kResampleThreads;
    resample_kernel<<<(unsigned)blocks, kResampleThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

}  // namespace sept
