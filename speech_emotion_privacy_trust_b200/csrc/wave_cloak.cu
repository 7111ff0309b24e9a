// Waveform-domain cloak: a learned noise of period L tiled over every utterance of a ragged batch (sm_100a).
//
//   wave_add_kernel     y[s] = x[s] + noise[(s - utt_off[u]) mod L] for every sample s of utterance u; samples before
//                       the first and after the last utterance are copied.  Each CTA owns one contiguous run of aligned
//                       quads; a thread finds its utterance once (binary search) and walks forward from there.  x and y
//                       move as float4 whatever the utterance alignment; the noise (L floats, L2-resident) is read as
//                       float4 when the quad's phase is a multiple of 4, else as scalars.  Quads that straddle an
//                       utterance boundary or the end of the buffer go sample by sample.
//   wave_reduce_kernel  backward, pass 1: r_s[j] = sum of g over the samples of phase j in slice s.  A tile is one
//                       period of one utterance (tile k of utterance u covers utt_off[u] + kL .. + L, clipped to the
//                       utterance); slice s owns the global tiles [n_tiles * s / S, n_tiles * (s+1) / S), S =
//                       kWaveSlices.  Tiles are staged 256 at a time (chunk); within a chunk, lane l of R sums the
//                       chunk's tiles l, l+R, ... in order, the lane sums are added in lane order, and the chunk sums
//                       are added to the slice's row in chunk order.  R = 1 when L/4 >= 256 quads, else 256 / (L/4).
//   wave_merge_kernel   backward, pass 2: r[j] = the slices summed in order: lane l of 8 sums slices 74l .. 74l+73 in
//                       order, the 8 lane sums are added in lane order.
//   wave_sigma_kernel   evaluation, pre-pass: sigma(rhos[j]) of the period into the caller's workspace, once per call.
//   wave_eval_add_kernel evaluation: y[s] = x[s] + (mu[j] + sigma[j] * eps_u[j]), j = (s - utt_off[u]) mod L, a fresh
//                       eps_u per utterance drawn inside the kernel (row d_u of sept_cloak_fwd_f32's per-sample draw);
//                       a thread walks the phase quads that start in its aligned quad, one normal4 per phase quad.
//   wave_reduce_per_utt_kernel  backward of the evaluation forward, pass 1: wave_reduce_kernel's rows of g and, in the
//                       same order, rows of g * eps_u (each eps_u drawn again inside the kernel, one normal4 per tile and
//                       phase quad, each product rounded on its own).
//   wave_merge_per_utt_kernel   pass 2: both row sets merged in wave_merge_kernel's order; dlocs, drhos = q * sigma'.
// No atomics: the order above is fixed, so the gradient is the same bits on every run (tests/wave_cloak_order.py
// restates it on the host).  The add and the backward are HBM-bound with no reuse of x, y or g.
#include <cuda_runtime.h>
#include <cstdint>

#include "cloak_noise.cuh"
#include "philox.cuh"
#include "wave_cloak.h"

namespace sept {

__device__ __forceinline__ float4 f4add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

__device__ __forceinline__ float& f4at(float4& v, int e) { return e == 0 ? v.x : e == 1 ? v.y : e == 2 ? v.z : v.w; }

// the last index u in [0, n - 1] with off[u] <= key (0 when n <= 1): the utterance (or tile run) holding key
__device__ __forceinline__ int last_le(const int64_t* off, int n, int64_t key) {
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= key) lo = mid; else hi = mid - 1;
    }
    return lo;
}

constexpr int kAddUnroll = 4;   // quads in flight per thread

__global__ void __launch_bounds__(kWaveThreads) wave_add_kernel(const WaveAddParams p) {
    const int64_t nq = (p.n + 3) / 4;
    const int64_t per = (nq + gridDim.x - 1) / gridDim.x;
    const int64_t q0 = (int64_t)blockIdx.x * per, q1 = q0 + per < nq ? q0 + per : nq;
    if (q0 + threadIdx.x >= q1) return;
    const int64_t lo = p.utt_off[0], hi = p.utt_off[p.n_utts];      // samples outside [lo, hi) are copied
    const uint32_t L = (uint32_t)p.period;
    int u = last_le(p.utt_off, p.n_utts, 4 * (q0 + threadIdx.x));
    int64_t b = 0, e = 0;                                           // bounds of utterance u (read once u is in range)
    bool have = false;
    for (int64_t qb = q0 + threadIdx.x; qb < q1; qb += kAddUnroll * kWaveThreads) {
        float4 v[kAddUnroll];
#pragma unroll
        for (int k = 0; k < kAddUnroll; ++k) {
            const int64_t q = qb + (int64_t)k * kWaveThreads;
            if (q < q1 && 4 * q + 4 <= p.n) v[k] = __ldcs(reinterpret_cast<const float4*>(p.x) + q);
        }
#pragma unroll
        for (int k = 0; k < kAddUnroll; ++k) {
            const int64_t q = qb + (int64_t)k * kWaveThreads;
            if (q >= q1) break;
            const int64_t s = 4 * q;
            if (s + 4 <= p.n && (s + 4 <= lo || s >= hi)) {            // wholly outside every utterance
                __stcs(reinterpret_cast<float4*>(p.y) + q, v[k]);
                continue;
            }
            if (s >= lo) {
                while (u + 1 < p.n_utts && p.utt_off[u + 1] <= s) { ++u; have = false; }
            }
            if (!have && p.n_utts > 0) { b = p.utt_off[u]; e = p.utt_off[u + 1]; have = true; }
            if (s + 4 <= p.n && s >= b && s + 4 <= e && have) {    // wholly inside utterance u
                const uint32_t ph = (uint32_t)(s - b) % L;
                float4 nz;
                if ((ph & 3u) == 0) {
                    nz = *reinterpret_cast<const float4*>(p.noise + ph);
                } else {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const uint32_t j = ph + c;
                        f4at(nz, c) = __ldg(p.noise + (j >= L ? j - L : j));
                    }
                }
                __stcs(reinterpret_cast<float4*>(p.y) + q, f4add(v[k], nz));
                continue;
            }
            // an utterance boundary, the edge of [lo, hi) or the end of the buffer lies inside this quad
            int w = u;
            for (int c = 0; c < 4 && s + c < p.n; ++c) {
                const int64_t t = s + c;
                float val = p.x[t];
                if (t >= lo && t < hi) {
                    while (w + 1 < p.n_utts && p.utt_off[w + 1] <= t) ++w;
                    val += __ldg(p.noise + (uint32_t)(t - p.utt_off[w]) % L);
                }
                p.y[t] = val;
            }
        }
    }
}

__global__ void __launch_bounds__(kWaveThreads) wave_sigma_kernel(const float* __restrict__ rhos, int L, float mn, float mx,
                                                                  float* __restrict__ sigma) {
    for (int j = blockIdx.x * kWaveThreads + threadIdx.x; j < L; j += gridDim.x * kWaveThreads) sigma[j] = sigma_of(rhos[j], mn, mx);
}

struct EvalUtt {
    int64_t b;               // first sample
    uint64_t ctr;            // Philox counter of phase quad 0: offset + draw index * L/4
    const float* eps;        // the caller's row, or null
};

__device__ __forceinline__ EvalUtt eval_utt(const WaveEvalParams& p, int u, uint64_t draw0) {
    const uint64_t d = draw0 + (p.utt_draw ? (uint64_t)p.utt_draw[u] : (uint64_t)u);
    return {p.utt_off[u], p.offset + d * (uint64_t)(p.period / 4), p.eps ? p.eps + (size_t)u * p.period : nullptr};
}

// mu + sigma * eps of the phases j .. j+3 (j a multiple of 4): one normal4, the same one sept_cloak_fwd_f32 draws for
// row d, elements j .. j+3
__device__ __forceinline__ float4 eval_noise4(const WaveEvalParams& p, const EvalUtt& t, uint32_t j) {
    const float4 e = t.eps ? __ldg(reinterpret_cast<const float4*>(t.eps + j)) : normal4(p.seed, t.ctr, j / 4, p.eps_std);
    const float4 mu = __ldg(reinterpret_cast<const float4*>(p.locs + j));
    const float4 sg = __ldg(reinterpret_cast<const float4*>(p.sigma + j));
    return make_float4(noise_of(mu.x, sg.x, e.x), noise_of(mu.y, sg.y, e.y), noise_of(mu.z, sg.z, e.z), noise_of(mu.w, sg.w, e.w));
}

// four consecutive samples at x + s, where s = a (mod 4) and x is 16-byte aligned
__device__ __forceinline__ float4 ld_quad(const float* x, int64_t s, int a) {
    if (a == 0) return __ldcs(reinterpret_cast<const float4*>(x + s));
    if (a == 2) {
        const float2 l = __ldcs(reinterpret_cast<const float2*>(x + s)), h = __ldcs(reinterpret_cast<const float2*>(x + s + 2));
        return make_float4(l.x, l.y, h.x, h.y);
    }
    return make_float4(__ldcs(x + s), __ldcs(x + s + 1), __ldcs(x + s + 2), __ldcs(x + s + 3));
}

__device__ __forceinline__ void st_quad(float* y, int64_t s, int a, float4 v) {
    if (a == 0) { __stcs(reinterpret_cast<float4*>(y + s), v); return; }
    if (a == 2) {
        __stcs(reinterpret_cast<float2*>(y + s), make_float2(v.x, v.y));
        __stcs(reinterpret_cast<float2*>(y + s + 2), make_float2(v.z, v.w));
        return;
    }
    __stcs(y + s, v.x); __stcs(y + s + 1, v.y); __stcs(y + s + 2, v.z); __stcs(y + s + 3, v.w);
}

constexpr int kEvalUnroll = 4;   // quads whose x is loaded before the first draw

// Thread q owns the phase quads that start in the aligned quad [4q, 4q + 4): utterance u's phase quad k covers samples
// b_u + 4k .. + 3 (clipped to the utterance), and exactly one of its samples 4q + (b_u & 3) lies in each aligned quad.
// So every in-utterance sample is written once, one normal4 per phase quad, and x / y are moved at the utterance's
// alignment (float4, two float2 or four floats).  The common case is a phase quad wholly inside the utterance that also
// covers the whole aligned quad; anything else (an utterance start, end or gap in the quad) goes to the general path.
__global__ void __launch_bounds__(kWaveThreads) wave_eval_add_kernel(const WaveEvalParams p) {
    const int64_t nq = (p.n + 3) / 4;
    const int64_t per = (nq + gridDim.x - 1) / gridDim.x;
    const int64_t q0 = (int64_t)blockIdx.x * per, q1 = q0 + per < nq ? q0 + per : nq;
    if (q0 + threadIdx.x >= q1) return;
    const int64_t lo = p.utt_off[0], hi = p.utt_off[p.n_utts];      // samples outside [lo, hi) are copied
    const uint32_t L = (uint32_t)p.period;
    const uint64_t draw0 = p.draw ? *p.draw : 0;
    int u = last_le(p.utt_off, p.n_utts, 4 * (q0 + threadIdx.x));
    int64_t b = 0, e = 0;                                           // bounds of utterance u (read once u is in range)
    bool have = false;
    int tu = -1;                                                    // the utterance t describes
    EvalUtt t{};
    for (int64_t qb = q0 + threadIdx.x; qb < q1; qb += kEvalUnroll * kWaveThreads) {
        float4 v[kEvalUnroll];
        int uk[kEvalUnroll];
        bool fast[kEvalUnroll];
#pragma unroll
        for (int k = 0; k < kEvalUnroll; ++k) {
            const int64_t q = qb + (int64_t)k * kWaveThreads, s0 = 4 * q;
            fast[k] = false;
            if (q >= q1) continue;
            if (s0 >= lo) {
                while (u + 1 < p.n_utts && p.utt_off[u + 1] <= s0) { ++u; have = false; }
            }
            if (!have && p.n_utts > 0) { b = p.utt_off[u]; e = p.utt_off[u + 1]; have = true; }
            uk[k] = u;
            const int a = (int)(b & 3);
            fast[k] = have && b <= s0 && s0 + a + 4 <= e;
            if (fast[k]) v[k] = ld_quad(p.x, s0 + a, a);
        }
#pragma unroll
        for (int k = 0; k < kEvalUnroll; ++k) {
            const int64_t q = qb + (int64_t)k * kWaveThreads, s0 = 4 * q;
            if (q >= q1) break;
            if (fast[k]) {
                if (uk[k] != tu) { t = eval_utt(p, uk[k], draw0); tu = uk[k]; }
                const int a = (int)(t.b & 3);
                const int64_t s = s0 + a;
                const float4 nz = eval_noise4(p, t, (uint32_t)(s - t.b) % L), x = v[k];
                st_quad(p.y, s, a, make_float4(__fadd_rn(x.x, nz.x), __fadd_rn(x.y, nz.y), __fadd_rn(x.z, nz.z), __fadd_rn(x.w, nz.w)));
                continue;
            }
            const int64_t s1 = s0 + 4 < p.n ? s0 + 4 : p.n;
            for (int64_t s = s0; s < s1; ++s)                       // samples outside every utterance
                if (s < lo || s >= hi) p.y[s] = p.x[s];
            for (int w = uk[k]; w < p.n_utts && p.utt_off[w] < s0 + 4; ++w) {   // phase quads starting in this quad
                const EvalUtt tw = eval_utt(p, w, draw0);
                const int64_t s = s0 + (tw.b & 3), ew = p.utt_off[w + 1];
                if (s < tw.b || s >= ew) continue;
                float4 nz = eval_noise4(p, tw, (uint32_t)(s - tw.b) % L);
                for (int c = 0; c < 4 && s + c < ew; ++c) p.y[s + c] = __fadd_rn(p.x[s + c], f4at(nz, c));
            }
        }
    }
}

__device__ __forceinline__ float4 tile_quad(const float* g, int64_t base, int len, int j) {
    if (j + 4 <= len && (base & 3) == 0) return __ldcs(reinterpret_cast<const float4*>(g + base + j));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int c = 0; c < 4; ++c)
        if (j + c < len) f4at(v, c) = __ldcs(g + base + j + c);
    return v;
}

__device__ __forceinline__ float4 f4mul(float4 a, float4 b) {                 // rounded on its own: no FMA into a sum
    return make_float4(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y), __fmul_rn(a.z, b.z), __fmul_rn(a.w, b.w));
}

// The per-utterance backward's staged tile data beyond base and length: the tile's Philox counter of phase quad 0
// (offset + d_u * L/4, the draw rule of eval_utt), or, with the caller's eps, the offset of its utterance's row.
__device__ __forceinline__ uint64_t* s_tile_ctr() { __shared__ uint64_t s[kWaveThreads]; return s; }
__device__ __forceinline__ float4* s_red_eps() { __shared__ float4 s[kWaveThreads]; return s; }

__device__ __forceinline__ uint64_t tile_ctr(const WaveReducePerUttParams& e, int u) {
    const int L = e.r.period;
    if (e.eps) return (uint64_t)u * L;
    const uint64_t d = (e.draw ? *e.draw : 0) + (e.utt_draw ? (uint64_t)e.utt_draw[u] : (uint64_t)u);
    return e.offset + d * (uint64_t)(L / 4);
}

// eps_u of the phases j .. j+3 (j a multiple of 4) of a tile: one normal4, the one wave_eval_add_kernel draws there
__device__ __forceinline__ float4 tile_eps(const WaveReducePerUttParams& e, uint64_t ctr, int j) {
    return e.eps ? __ldg(reinterpret_cast<const float4*>(e.eps + ctr + j)) : normal4(e.seed, ctr, (uint32_t)j / 4, e.eps_std);
}

// Backward pass 1 of slice blockIdx.x: the row of g (and, kEps, the row of g * eps_u, in the same order; a quad past
// the tile's end adds nothing to it, as +0 would not).
template <bool kEps>
__device__ __forceinline__ void reduce_slice(const WaveReduceParams& p, const WaveReducePerUttParams* e) {
    __shared__ int64_t s_base[kWaveThreads];
    __shared__ int s_len[kWaveThreads];
    __shared__ float4 s_red[kWaveThreads];
    const int L = p.period, Q = L / 4;
    const int R = Q >= kWaveThreads ? 1 : kWaveThreads / Q;
    const int lane = R == 1 ? 0 : threadIdx.x / Q;
    const int qt = R == 1 ? threadIdx.x : threadIdx.x % Q;
    const int64_t T0 = p.n_tiles * blockIdx.x / kWaveSlices, T1 = p.n_tiles * (blockIdx.x + 1) / kWaveSlices;
    float* row = p.partial + (size_t)blockIdx.x * L;
    float* row_e = kEps ? p.partial + (size_t)(kWaveSlices + blockIdx.x) * L : nullptr;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    if (T0 == T1) {                                                 // an empty slice still writes its (zero) row
        if (lane == 0)
            for (int q = qt; q < Q; q += kWaveThreads) {
                *reinterpret_cast<float4*>(row + 4 * q) = zero;
                if constexpr (kEps) *reinterpret_cast<float4*>(row_e + 4 * q) = zero;
            }
        return;
    }
    float4 acc = zero, acc_e = zero;                                // R > 1: the row elements of quad qt
    for (int64_t c0 = T0; c0 < T1; c0 += kWaveThreads) {
        const int nt = T1 - c0 < kWaveThreads ? (int)(T1 - c0) : kWaveThreads;
        __syncthreads();                                            // the previous chunk is no longer read
        if ((int)threadIdx.x < nt) {
            const int64_t i = c0 + threadIdx.x;
            const int u = last_le(p.tile_off, p.n_utts, i);
            const int64_t base = p.utt_off[u] + (i - p.tile_off[u]) * L, left = p.utt_off[u + 1] - base;
            s_base[threadIdx.x] = base;
            s_len[threadIdx.x] = left < L ? (int)left : L;
            if constexpr (kEps) s_tile_ctr()[threadIdx.x] = tile_ctr(*e, u);
        }
        __syncthreads();
        if (R == 1) {
            for (int q = qt; q < Q; q += kWaveThreads) {
                float4 l = zero, le = zero;
#pragma unroll 8
                for (int t = 0; t < nt; ++t) {
                    const float4 gq = tile_quad(p.g, s_base[t], s_len[t], 4 * q);
                    l = f4add(l, gq);
                    if constexpr (kEps)
                        if (4 * q < s_len[t]) le = f4add(le, f4mul(gq, tile_eps(*e, s_tile_ctr()[t], 4 * q)));
                }
                float4* dst = reinterpret_cast<float4*>(row + 4 * q);
                *dst = f4add(c0 == T0 ? zero : *dst, l);
                if constexpr (kEps) {
                    float4* dst_e = reinterpret_cast<float4*>(row_e + 4 * q);
                    *dst_e = f4add(c0 == T0 ? zero : *dst_e, le);
                }
            }
        } else {
            float4 l = zero, le = zero;
            if (lane < R)
                for (int t = lane; t < nt; t += R) {
                    const float4 gq = tile_quad(p.g, s_base[t], s_len[t], 4 * qt);
                    l = f4add(l, gq);
                    if constexpr (kEps)
                        if (4 * qt < s_len[t]) le = f4add(le, f4mul(gq, tile_eps(*e, s_tile_ctr()[t], 4 * qt)));
                }
            s_red[threadIdx.x] = l;
            if constexpr (kEps) s_red_eps()[threadIdx.x] = le;
            __syncthreads();
            if (lane == 0) {
                float4 c = s_red[qt];
                for (int k = 1; k < R; ++k) c = f4add(c, s_red[k * Q + qt]);
                acc = f4add(acc, c);
                if constexpr (kEps) {
                    const float4* se = s_red_eps();
                    float4 ce = se[qt];
                    for (int k = 1; k < R; ++k) ce = f4add(ce, se[k * Q + qt]);
                    acc_e = f4add(acc_e, ce);
                }
            }
        }
    }
    if (R > 1 && lane == 0) {
        *reinterpret_cast<float4*>(row + 4 * qt) = acc;
        if constexpr (kEps) *reinterpret_cast<float4*>(row_e + 4 * qt) = acc_e;
    }
}

__global__ void __launch_bounds__(kWaveThreads) wave_reduce_kernel(const WaveReduceParams p) {
    reduce_slice<false>(p, nullptr);
}

__global__ void __launch_bounds__(kWaveThreads) wave_reduce_per_utt_kernel(const __grid_constant__ WaveReducePerUttParams p) {
    reduce_slice<true>(p.r, &p);
}

constexpr int kMergeQuads = kWaveThreads / kWaveMergeLanes;        // 32 quads per CTA
static_assert(kWaveSlices % kWaveMergeLanes == 0, "equal slice runs per merge lane");

// Backward pass 2 at quad q of the period: the kWaveSlices rows at `partial` summed in order, valid in lane 0.  Every
// thread of the CTA calls it (it synchronises); s_red is the caller's shared scratch of kWaveThreads quads.
__device__ __forceinline__ float4 merge_quad(const float* __restrict__ partial, int L, int q, float4* s_red) {
    const int Q = L / 4, lane = threadIdx.x / kMergeQuads, qi = threadIdx.x % kMergeQuads;
    constexpr int per = kWaveSlices / kWaveMergeLanes;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q < Q) {
#pragma unroll 8
        for (int s = lane * per; s < (lane + 1) * per; ++s)
            a = f4add(a, __ldcg(reinterpret_cast<const float4*>(partial + (size_t)s * L) + q));
    }
    s_red[threadIdx.x] = a;
    __syncthreads();
    float4 c = a;
    if (lane == 0 && q < Q) {
        c = s_red[qi];
        for (int k = 1; k < kWaveMergeLanes; ++k) c = f4add(c, s_red[k * kMergeQuads + qi]);
    }
    return c;
}

__global__ void __launch_bounds__(kWaveThreads) wave_merge_kernel(const float* __restrict__ partial, int L,
                                                                  float* __restrict__ r) {
    __shared__ float4 s_red[kWaveThreads];
    const int q = blockIdx.x * kMergeQuads + threadIdx.x % kMergeQuads;
    const float4 c = merge_quad(partial, L, q, s_red);
    if (threadIdx.x < kMergeQuads && q < L / 4) reinterpret_cast<float4*>(r)[q] = c;
}

// dlocs = the merged rows of g; drhos = the merged rows of g * eps_u times sigma'(rho), rounded on its own
__global__ void __launch_bounds__(kWaveThreads) wave_merge_per_utt_kernel(const float* __restrict__ partial, int L,
                                                                          const float* __restrict__ rhos, float mn,
                                                                          float mx, float* __restrict__ dlocs,
                                                                          float* __restrict__ drhos) {
    __shared__ float4 s_red[kWaveThreads], s_red_e[kWaveThreads];
    const int q = blockIdx.x * kMergeQuads + threadIdx.x % kMergeQuads;
    const float4 c = merge_quad(partial, L, q, s_red);
    const float4 w = merge_quad(partial + (size_t)kWaveSlices * L, L, q, s_red_e);
    if (threadIdx.x < kMergeQuads && q < L / 4) {
        reinterpret_cast<float4*>(dlocs)[q] = c;
        const float4 rho = __ldg(reinterpret_cast<const float4*>(rhos) + q);
        reinterpret_cast<float4*>(drhos)[q] = f4mul(w, make_float4(dsigma_of(rho.x, mn, mx), dsigma_of(rho.y, mn, mx),
                                                                   dsigma_of(rho.z, mn, mx), dsigma_of(rho.w, mn, mx)));
    }
}

cudaError_t launch_wave_add(const WaveAddParams& p, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int64_t nq = (p.n + 3) / 4, want = (nq + kAddUnroll * kWaveThreads - 1) / (kAddUnroll * kWaveThreads);
    const int blocks = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);     // 8 CTAs (2048 threads) per SM
    wave_add_kernel<<<blocks, kWaveThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_wave_eval(const WaveEvalParams& p, cudaStream_t stream) {
    if (p.n == 0) return cudaSuccess;
    int dev = 0, sms = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    const int sb = (p.period + kWaveThreads - 1) / kWaveThreads;
    wave_sigma_kernel<<<sb < sms ? sb : sms, kWaveThreads, 0, stream>>>(p.rhos, p.period, p.min_scale, p.max_scale, p.sigma);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int64_t nq = (p.n + 3) / 4, want = (nq + kEvalUnroll * kWaveThreads - 1) / (kEvalUnroll * kWaveThreads);
    const int blocks = (int)(want < (int64_t)sms * 8 ? want : (int64_t)sms * 8);
    wave_eval_add_kernel<<<blocks, kWaveThreads, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_wave_reduce(const WaveReduceParams& p, cudaStream_t stream) {
    wave_reduce_kernel<<<kWaveSlices, kWaveThreads, 0, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int quads = p.period / 4;
    wave_merge_kernel<<<(quads + kMergeQuads - 1) / kMergeQuads, kWaveThreads, 0, stream>>>(p.partial, p.period, p.r);
    return cudaGetLastError();
}

cudaError_t launch_wave_reduce_per_utt(const WaveReducePerUttParams& p, cudaStream_t stream) {
    wave_reduce_per_utt_kernel<<<kWaveSlices, kWaveThreads, 0, stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const int quads = p.r.period / 4;
    wave_merge_per_utt_kernel<<<(quads + kMergeQuads - 1) / kMergeQuads, kWaveThreads, 0, stream>>>(
        p.r.partial, p.r.period, p.rhos, p.min_scale, p.max_scale, p.r.r, p.drhos);
    return cudaGetLastError();
}

}  // namespace sept
