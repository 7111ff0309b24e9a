// Per-speaker feature statistics and normalisation (sm_100a).
//
// The reference appends every frame of every training window to a per-speaker Python list and reduces it with
// numpy (preprocess_data/preprocess_adversary_data.py:26-27, 41-48, 357-364): a frame that lies in k overlapping
// windows is counted k times.  Here the multiplicity is a closed-form weight and the statistics are weighted
// Welford accumulations: one CTA per utterance (thread = feature, coalesced rows), then one CTA per speaker merges
// its utterances' partials with Chan's formula in list order (deterministic, no atomics).
// Features of width 128 (the reference's, training_data_preprocess.sh --input_spec_size 128) take vectorised paths.
//   znorm   (x - mean) / (std + 1e-5)            :378
//   min_max (x - min) / (max - min) * 2 - 1      :380
#include <cuda_runtime.h>
#include <cfloat>
#include <cstdint>

#include "norm.h"
#include "norm_weight.cuh"

namespace sept {

__global__ void __launch_bounds__(128) utt_partial_kernel(const SpeakerStatsParams p) {
    const int u = blockIdx.x;
    const long long f0 = p.frame_off[u];
    const int T = (int)(p.frame_off[u + 1] - f0);
    const bool whole = p.whole ? p.whole[u] != 0 : false;
    const int F = p.n_feat;
    for (int f = threadIdx.x; f < F; f += blockDim.x) {
        float n = 0.f, mean = 0.f, m2 = 0.f, mn = FLT_MAX, mx = -FLT_MAX;
        const float* col = p.feat + f0 * F + f;
        for (int t = 0; t < T; ++t) {
            const int w = frame_weight(t, T, p.win_len, p.shift_len, whole);
            if (w == 0) continue;
            const float x = col[(long long)t * F];
            n += (float)w;
            const float d = x - mean;
            mean += d * ((float)w / n);
            m2 += (float)w * d * (x - mean);
            mn = fminf(mn, x);
            mx = fmaxf(mx, x);
        }
        float* o = p.utt_partial + ((long long)u * kStatRows) * F + f;
        o[0] = n; o[F] = mean; o[2 * F] = m2; o[3 * F] = mn; o[4 * F] = mx;
    }
}

// F == 128 fast path: 8 warps per utterance, warp w takes frames t = w, w+8, ...; a lane owns 4 adjacent features, so
// every frame row is one coalesced 512-byte warp load and four rows are in flight per lane.  The warps' partials are
// merged in warp order (Chan), which keeps the result deterministic.
struct Welford4 {
    float n;
    float4 mean, m2, mn, mx;
};

__device__ __forceinline__ void welford_add(float& mean, float& m2, float& mn, float& mx, float x, float w, float r) {
    const float d = x - mean;
    mean += d * r;                                              // r = w / n_new
    m2 += w * d * (x - mean);
    mn = fminf(mn, x);
    mx = fmaxf(mx, x);
}

__device__ __forceinline__ void chan_merge(float& n, float& mean, float& m2, float nb, float mb, float m2b) {
    const float tot = n + nb, d = mb - mean;
    mean += d * (nb / tot);
    m2 += m2b + d * d * (n * nb / tot);
}

__global__ void __launch_bounds__(256) utt_partial128_kernel(const SpeakerStatsParams p) {
    constexpr int F = 128, WARPS = 8;
    __shared__ float sh[WARPS][4][F];                             // mean, m2, min, max per warp
    __shared__ float sh_n[WARPS];
    const int u = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long f0 = p.frame_off[u];
    const int T = (int)(p.frame_off[u + 1] - f0);
    const bool whole = p.whole ? p.whole[u] != 0 : false;
    const float4* rows = reinterpret_cast<const float4*>(p.feat + f0 * F) + lane;
    float n = 0.f;
    float4 mean = make_float4(0.f, 0.f, 0.f, 0.f), m2 = mean;
    float4 mn = make_float4(FLT_MAX, FLT_MAX, FLT_MAX, FLT_MAX), mx = make_float4(-FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX);
    const float inv_shift = 1.0f / (float)p.shift_len;
    const int n_win = T >= p.win_len ? (T - p.win_len) / p.shift_len + 1 : 0;
    for (int t = warp; t < T; t += 4 * WARPS) {
        float4 x[4];
        int w[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int tt = t + j * WARPS;
            w[j] = tt < T ? frame_weight_fast(tt, T, p.win_len, p.shift_len, inv_shift, n_win, whole) : 0;
            if (w[j]) x[j] = rows[(long long)tt * (F / 4)];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (!w[j]) continue;
            const float wf = (float)w[j];
            n += wf;
            const float r = __fdividef(wf, n);                    // 2 ulp; n <= 4 T, far from the fast division's range limit
            welford_add(mean.x, m2.x, mn.x, mx.x, x[j].x, wf, r);
            welford_add(mean.y, m2.y, mn.y, mx.y, x[j].y, wf, r);
            welford_add(mean.z, m2.z, mn.z, mx.z, x[j].z, wf, r);
            welford_add(mean.w, m2.w, mn.w, mx.w, x[j].w, wf, r);
        }
    }
    reinterpret_cast<float4*>(sh[warp][0])[lane] = mean;
    reinterpret_cast<float4*>(sh[warp][1])[lane] = m2;
    reinterpret_cast<float4*>(sh[warp][2])[lane] = mn;
    reinterpret_cast<float4*>(sh[warp][3])[lane] = mx;
    if (lane == 0) sh_n[warp] = n;
    __syncthreads();
    if (threadIdx.x < F) {
        const int f = threadIdx.x;
        float tn = 0.f, tm = 0.f, t2 = 0.f, tmin = FLT_MAX, tmax = -FLT_MAX;
        for (int w = 0; w < WARPS; ++w) {
            const float nb = sh_n[w];
            if (nb == 0.f) continue;
            chan_merge(tn, tm, t2, nb, sh[w][0][f], sh[w][1][f]);
            tn += nb;
            tmin = fminf(tmin, sh[w][2][f]);
            tmax = fmaxf(tmax, sh[w][3][f]);
        }
        float* o = p.utt_partial + ((long long)u * kStatRows) * F + f;
        o[0] = tn; o[F] = tm; o[2 * F] = t2; o[3 * F] = tmin; o[4 * F] = tmax;
    }
}

// one CTA per speaker: 8 slices of 128 feature-threads walk the speaker's utterance list interleaved (slice s takes
// entries s, s+8, ...), then slice 0 folds the 8 partials in slice order -- deterministic, no atomics
constexpr int kMergeSlices = 8;

__global__ void __launch_bounds__(128 * kMergeSlices) speaker_merge_kernel(const SpeakerStatsParams p) {
    __shared__ float sh[kMergeSlices][kStatRows][128];
    const int s = blockIdx.x, F = p.n_feat;
    const int fl = threadIdx.x & 127, slice = threadIdx.x >> 7;
    const int j0 = p.spk_ptr[s], j1 = p.spk_ptr[s + 1];
    for (int fbase = 0; fbase < F; fbase += 128) {
        const int f = fbase + fl;
        float n = 0.f, mean = 0.f, m2 = 0.f, mn = FLT_MAX, mx = -FLT_MAX;
        if (f < F) {
            for (int j = j0 + slice; j < j1; j += kMergeSlices) {
                const float* o = p.utt_partial + ((long long)p.spk_utts[j] * kStatRows) * F + f;
                const float nb = o[0];
                if (nb == 0.f) continue;
                chan_merge(n, mean, m2, nb, o[F], o[2 * F]);
                n += nb;
                mn = fminf(mn, o[3 * F]);
                mx = fmaxf(mx, o[4 * F]);
            }
        }
        sh[slice][0][fl] = n; sh[slice][1][fl] = mean; sh[slice][2][fl] = m2; sh[slice][3][fl] = mn; sh[slice][4][fl] = mx;
        __syncthreads();
        if (slice == 0 && f < F) {
            n = 0.f; mean = 0.f; m2 = 0.f; mn = FLT_MAX; mx = -FLT_MAX;
            for (int k = 0; k < kMergeSlices; ++k) {
                const float nb = sh[k][0][fl];
                if (nb == 0.f) continue;
                chan_merge(n, mean, m2, nb, sh[k][1][fl], sh[k][2][fl]);
                n += nb;
                mn = fminf(mn, sh[k][3][fl]);
                mx = fmaxf(mx, sh[k][4][fl]);
            }
            float* r = p.stats + ((long long)s * kStatRows) * F + f;
            r[0] = n; r[F] = mean; r[2 * F] = n > 0.f ? sqrtf(m2 / n) : 0.f; r[3 * F] = mn; r[4 * F] = mx;
        }
        __syncthreads();
    }
}

// z = fmaf(x - a, b, c): znorm a = mean, b = 1 / (std + 1e-5), c = 0; min_max a = min, b = 2 / (max - min), c = -1.
// Both normalisation kernels (and the backward, norm_bwd.cu) evaluate this one expression, so the kernel a call takes
// (F, pointer alignment) does not change a bit of its result.
__device__ __forceinline__ void norm_coef(int mode, float mean, float sd, float mn, float mx, float& a, float& b) {
    if (mode == 0) { a = mean; b = 1.0f / (sd + 1e-5f); }
    else { a = mn; b = 2.0f / (mx - mn); }
}

__device__ __forceinline__ float norm_c(int mode) { return mode == 0 ? 0.f : -1.f; }

__global__ void __launch_bounds__(256) normalize_kernel(const NormalizeParams p) {
    const int F = p.n_feat;
    int u, t_begin, rows, T;
    float* out;
    if (p.win_utt) {
        u = p.win_utt[blockIdx.x];
        t_begin = p.win_t0[blockIdx.x];
        rows = p.win_len;
        out = p.out + (long long)blockIdx.x * p.win_len * F;
    } else {
        u = blockIdx.x;
        t_begin = 0;
        rows = (int)(p.frame_off[u + 1] - p.frame_off[u]);
        out = p.out + p.frame_off[u] * F;
    }
    const long long f0 = p.frame_off[u];
    T = (int)(p.frame_off[u + 1] - f0);
    const float* st = p.stats + ((long long)p.spk_of_utt[u] * kStatRows) * F;
    const int total = rows * F;
    const float c = norm_c(p.mode);
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        const int r = i / F, f = i - r * F;
        const int t = t_begin + r;
        const float x = t < T ? p.feat[(f0 + t) * F + f] : 0.f;
        float a, b;
        norm_coef(p.mode, st[F + f], st[2 * F + f], st[3 * F + f], st[4 * F + f], a, b);
        out[i] = fmaf(x - a, b, c);
    }
}

// n_feat % 4 == 0: a thread owns 4 adjacent features of a row; rows are coalesced 16-byte accesses
__global__ void __launch_bounds__(256) normalize4_kernel(const NormalizeParams p) {
    const int F4 = p.n_feat / 4;
    int u, t_begin, rows;
    float4* out;
    if (p.win_utt) {
        u = p.win_utt[blockIdx.x];
        t_begin = p.win_t0[blockIdx.x];
        rows = p.win_len;
        out = reinterpret_cast<float4*>(p.out + (long long)blockIdx.x * p.win_len * p.n_feat);
    } else {
        u = blockIdx.x;
        t_begin = 0;
        rows = (int)(p.frame_off[u + 1] - p.frame_off[u]);
        out = reinterpret_cast<float4*>(p.out + p.frame_off[u] * p.n_feat);
    }
    const long long f0 = p.frame_off[u];
    const int T = (int)(p.frame_off[u + 1] - f0);
    const float* st = p.stats + ((long long)p.spk_of_utt[u] * kStatRows) * p.n_feat;
    const float4* in = reinterpret_cast<const float4*>(p.feat + f0 * p.n_feat);
    const int rows_per_pass = blockDim.x / F4 > 0 ? blockDim.x / F4 : 1;
    const int q = threadIdx.x % F4, r0 = threadIdx.x / F4;
    if (r0 >= rows_per_pass) return;
    const float4 mean = reinterpret_cast<const float4*>(st + p.n_feat)[q], sd = reinterpret_cast<const float4*>(st + 2 * p.n_feat)[q];
    const float4 mn = reinterpret_cast<const float4*>(st + 3 * p.n_feat)[q], mx = reinterpret_cast<const float4*>(st + 4 * p.n_feat)[q];
    // the divisions of norm_coef are done once per thread; four rows are in flight per thread
    float4 a, b;
    const float c = norm_c(p.mode);
    norm_coef(p.mode, mean.x, sd.x, mn.x, mx.x, a.x, b.x);
    norm_coef(p.mode, mean.y, sd.y, mn.y, mx.y, a.y, b.y);
    norm_coef(p.mode, mean.z, sd.z, mn.z, mx.z, a.z, b.z);
    norm_coef(p.mode, mean.w, sd.w, mn.w, mx.w, a.w, b.w);
    for (int r = r0; r < rows; r += 4 * rows_per_pass) {
        float4 x[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int rr = r + j * rows_per_pass, t = t_begin + rr;
            x[j] = (rr < rows && t < T) ? in[(long long)t * F4 + q] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int rr = r + j * rows_per_pass;
            if (rr >= rows) break;
            float4 z;
            z.x = fmaf(x[j].x - a.x, b.x, c); z.y = fmaf(x[j].y - a.y, b.y, c);
            z.z = fmaf(x[j].z - a.z, b.z, c); z.w = fmaf(x[j].w - a.w, b.w, c);
            out[(long long)rr * F4 + q] = z;
        }
    }
}

static bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

cudaError_t launch_speaker_stats(const SpeakerStatsParams& p, cudaStream_t stream) {
    if (p.n_utts > 0) {
        // float4 rows: feat + f0 * 128 is 16-byte aligned for every utterance exactly when feat is
        if (p.n_feat == 128 && aligned16(p.feat)) utt_partial128_kernel<<<p.n_utts, 256, 0, stream>>>(p);
        else utt_partial_kernel<<<p.n_utts, 128, 0, stream>>>(p);
    }
    if (p.n_spk > 0) speaker_merge_kernel<<<p.n_spk, 128 * kMergeSlices, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_normalize(const NormalizeParams& p, cudaStream_t stream) {
    const int blocks = p.win_utt ? p.n_windows : p.n_utts;
    if (blocks > 0) {
        const bool vec = p.n_feat % 4 == 0 && p.n_feat / 4 <= 256 && aligned16(p.feat) && aligned16(p.out) &&
                         aligned16(p.stats);
        if (vec) normalize4_kernel<<<blocks, 256, 0, stream>>>(p);
        else normalize_kernel<<<blocks, 256, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

}  // namespace sept
