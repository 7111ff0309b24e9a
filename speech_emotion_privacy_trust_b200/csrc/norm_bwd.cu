// Backward of the per-speaker statistics and normalisation (sm_100a): what torch autograd gives through the reference's
// own computation (preprocess_data/preprocess_adversary_data.py:26-27, 29-35, 357-385), where every window's rows are
// stacked per speaker with duplicates, reduced with mean / std / min / max, and the windows normalised and zero padded.
//
// Normalisation (z = (x - a) * b + c; znorm a = mean, b = 1 / (std + 1e-5), c = 0; min_max a = min, b = 2 / (max - min),
// c = -1), upstream gradient Zbar over every row of every window:
//   dx_t    = b * sum_{windows w containing t} Zbar[w, t - t0_w]
//   S1 = sum Zbar, S2 = sum Zbar * z over the speaker's rows, padded rows included (their z = (0 - a) * b + c)
//   znorm   d mean = -b S1, d std = -b S2;   min_max  d min = b (S2 - S1) / 2, d max = -b (S2 + S1) / 2
// Statistics (w_t = training-window multiplicity of frame t, N = sum w_t):
//   dx_t += w_t d mean / N + w_t (x_t - mean) / (N std) d std          (no std term where the forward's std is exactly 0)
//        +  w_t / W_min d min   if x_t == min  (W_min = sum of w over the speaker's frames equal to min; max alike)
// Frames with w_t = 0 get no statistics gradient.  Every pass is one CTA per utterance (frames walked in a fixed
// order) or one CTA per speaker (utterances merged in list order): deterministic, no atomics.
#include <cuda_runtime.h>
#include <cstdint>

#include "norm_bwd.h"
#include "norm_weight.cuh"

namespace sept {

namespace {

constexpr int kBwdThreads = 256;
constexpr int kBwdMergeSlices = 8;

// Thread mapping of the per-utterance passes: a thread owns V adjacent features (column q of cols = F / V).  When a row
// has fewer columns than the CTA has threads, `groups` frames are walked at once (group g takes frames g, g + groups,
// ...) and the groups' partial sums are merged in group order; otherwise a thread walks every frame for columns
// q, q + 256, ...
struct RowMap {
    int cols, groups, g, q0, dq;
    __device__ RowMap(int F, int V) {
        cols = F / V;
        if (cols < kBwdThreads) {
            groups = kBwdThreads / cols; g = threadIdx.x / cols; q0 = threadIdx.x % cols; dq = cols;
        } else {
            groups = 1; g = 0; q0 = threadIdx.x; dq = kBwdThreads;
        }
    }
    __device__ bool active() const { return g < groups; }
};

template <int V>
__device__ __forceinline__ void ldv(float (&d)[V], const float* p) {
    if constexpr (V == 4) {
        const float4 q = *reinterpret_cast<const float4*>(p);
        d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
    } else {
#pragma unroll
        for (int i = 0; i < V; ++i) d[i] = p[i];
    }
}

template <int V>
__device__ __forceinline__ void addv(float (&d)[V], const float* p) {
    float x[V];
    ldv<V>(x, p);
#pragma unroll
    for (int i = 0; i < V; ++i) d[i] += x[i];
}

template <int V>
__device__ __forceinline__ void stv(float* p, const float (&d)[V]) {
    if constexpr (V == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(d[0], d[1], d[2], d[3]);
    } else {
#pragma unroll
        for (int i = 0; i < V; ++i) p[i] = d[i];
    }
}

// a CTA of kBwdMergeSlices x 128 threads sums rows [0, 2F) of the speaker's (2, F) utterance partials: slice k takes
// list entries k, k + 8, ... and slice 0 folds the slices in order.  Returns the sums of feature f in slice 0.
template <class T>
__device__ __forceinline__ void speaker_sum2(const T* part, const int32_t* spk_ptr, const int32_t* spk_utts, int s, int F,
                                             int f, T (&sh)[kBwdMergeSlices][2][128], T& r0, T& r1) {
    const int fl = threadIdx.x & 127, slice = threadIdx.x >> 7;
    T a0 = 0, a1 = 0;
    if (f < F) {
        for (int j = spk_ptr[s] + slice; j < spk_ptr[s + 1]; j += kBwdMergeSlices) {
            const T* o = part + (long long)spk_utts[j] * 2 * F + f;
            a0 += o[0];
            a1 += o[F];
        }
    }
    sh[slice][0][fl] = a0;
    sh[slice][1][fl] = a1;
    __syncthreads();
    r0 = 0; r1 = 0;
    if (slice == 0) {
        for (int k = 0; k < kBwdMergeSlices; ++k) {
            r0 += sh[k][0][fl];
            r1 += sh[k][1][fl];
        }
    }
    __syncthreads();
}

}  // namespace

// Pass 1: one CTA per utterance walks its frames; for frame t the rows of the windows covering it are the contiguous
// range [lo, hi) of the utterance's window list (sorted by t0), so every element of Zbar is read once.  Writes dfeat and
// the utterance's (S1, S2) partials, the padded rows of its windows included.
template <int V>
__global__ void __launch_bounds__(kBwdThreads) normalize_bwd_kernel(const NormalizeBwdParams p) {
    __shared__ float sh[2][kBwdThreads * V];
    const int F = p.f.n_feat, u = blockIdx.x, L = p.f.win_len;
    const RowMap m(F, V);
    const long long f0 = p.f.frame_off[u];
    const int T = (int)(p.f.frame_off[u + 1] - f0);
    const bool window = p.f.win_utt != nullptr, stats = p.upart != nullptr;
    const int j0 = window ? p.utt_win_ptr[u] : 0, j1 = window ? p.utt_win_ptr[u + 1] : 0;
    const float* st = p.f.stats + (long long)p.f.spk_of_utt[u] * kStatRows * F;
    if (m.active()) {
        for (int q = m.q0; q < m.cols; q += m.dq) {
            const int c = q * V;
            float a[V], b[V], s1[V], s2[V];
            const float cz = p.f.mode == 0 ? 0.f : -1.f;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                if (p.f.mode == 0) {
                    a[i] = st[F + c + i];
                    b[i] = 1.0f / (st[2 * F + c + i] + 1e-5f);
                } else {
                    a[i] = st[3 * F + c + i];
                    b[i] = 2.0f / (st[4 * F + c + i] - st[3 * F + c + i]);
                }
                s1[i] = 0.f; s2[i] = 0.f;
            }
            int lo = j0, hi = j0;
            for (int t = m.g; t < T; t += m.groups) {
                float gz[V];
#pragma unroll
                for (int i = 0; i < V; ++i) gz[i] = 0.f;
                if (window) {
                    while (hi < j1 && p.f.win_t0[p.utt_win[hi]] <= t) ++hi;
                    while (lo < hi && p.f.win_t0[p.utt_win[lo]] + L <= t) ++lo;
                    for (int j = lo; j < hi; ++j) {
                        const int w = p.utt_win[j];
                        addv<V>(gz, p.grad + ((long long)w * L + (t - p.f.win_t0[w])) * F + c);
                    }
                } else {
                    addv<V>(gz, p.grad + (f0 + t) * F + c);
                }
                if (p.dfeat) {
                    float d[V];
#pragma unroll
                    for (int i = 0; i < V; ++i) d[i] = gz[i] * b[i];
                    stv<V>(p.dfeat + (f0 + t) * F + c, d);
                }
                if (stats) {
                    float x[V];
                    ldv<V>(x, p.f.feat + (f0 + t) * F + c);
#pragma unroll
                    for (int i = 0; i < V; ++i) {
                        s1[i] += gz[i];
                        s2[i] = fmaf(gz[i], fmaf(x[i] - a[i], b[i], cz), s2[i]);
                    }
                }
            }
            if (!stats) continue;
            if (window) {                       // rows past the utterance end: the normalised zero padding of :29-35
                float ps[V];
#pragma unroll
                for (int i = 0; i < V; ++i) ps[i] = 0.f;
                for (int j = j0; j < j1; ++j) {
                    const int w = p.utt_win[j], t0 = p.f.win_t0[w];
                    for (int r = (T > t0 ? T - t0 : 0) + m.g; r < L; r += m.groups)
                        addv<V>(ps, p.grad + ((long long)w * L + r) * F + c);
                }
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    s1[i] += ps[i];
                    s2[i] = fmaf(ps[i], fmaf(0.f - a[i], b[i], cz), s2[i]);
                }
            }
            if (m.groups == 1) {
                float* o = p.upart + (long long)u * 2 * F + c;
#pragma unroll
                for (int i = 0; i < V; ++i) { o[i] = s1[i]; o[F + i] = s2[i]; }
            } else {
#pragma unroll
                for (int i = 0; i < V; ++i) { sh[0][m.g * F + c + i] = s1[i]; sh[1][m.g * F + c + i] = s2[i]; }
            }
        }
    }
    if (stats && m.groups > 1) {
        __syncthreads();
        if (threadIdx.x < m.cols) {
            const int c = threadIdx.x * V;
            float* o = p.upart + (long long)u * 2 * F + c;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                float r1 = 0.f, r2 = 0.f;
                for (int k = 0; k < m.groups; ++k) { r1 += sh[0][k * F + c + i]; r2 += sh[1][k * F + c + i]; }
                o[i] = r1; o[F + i] = r2;
            }
        }
    }
}

// Pass 2: one CTA per speaker merges its utterances' (S1, S2) in list order and writes d stats.
__global__ void __launch_bounds__(128 * kBwdMergeSlices) normalize_bwd_merge_kernel(const NormalizeBwdParams p) {
    __shared__ float sh[kBwdMergeSlices][2][128];
    const int s = blockIdx.x, F = p.f.n_feat;
    for (int fbase = 0; fbase < F; fbase += 128) {
        const int f = fbase + (threadIdx.x & 127);
        float S1, S2;
        speaker_sum2<float>(p.upart, p.spk_ptr, p.spk_utts, s, F, f, sh, S1, S2);
        if (threadIdx.x < 128 && f < F) {
            const float* st = p.f.stats + (long long)s * kStatRows * F + f;
            float* d = p.dstats + (long long)s * kStatRows * F + f;
            d[0] = 0.f;
            if (p.f.mode == 0) {
                const float b = 1.0f / (st[2 * F] + 1e-5f);
                d[F] = -b * S1; d[2 * F] = -b * S2; d[3 * F] = 0.f; d[4 * F] = 0.f;
            } else {
                const float b = 2.0f / (st[4 * F] - st[3 * F]);
                d[F] = 0.f; d[2 * F] = 0.f; d[3 * F] = 0.5f * b * (S2 - S1); d[4 * F] = -0.5f * b * (S2 + S1);
            }
        }
    }
}

// Statistics pass 1: per utterance and feature, the summed weight of the frames equal to the speaker's min / max
// (exact integers).
template <int V>
__global__ void __launch_bounds__(kBwdThreads) stats_bwd_ties_kernel(const SpeakerStatsBwdParams p) {
    __shared__ int sh[2][kBwdThreads * V];
    const int F = p.f.n_feat, u = blockIdx.x;
    const RowMap m(F, V);
    const long long f0 = p.f.frame_off[u];
    const int T = (int)(p.f.frame_off[u + 1] - f0);
    const bool whole = p.f.whole ? p.f.whole[u] != 0 : false;
    const float inv_shift = 1.0f / (float)p.f.shift_len;
    const int n_win = T >= p.f.win_len ? (T - p.f.win_len) / p.f.shift_len + 1 : 0;
    const float* st = p.f.stats + (long long)p.spk_of_utt[u] * kStatRows * F;
    if (m.active()) {
        for (int q = m.q0; q < m.cols; q += m.dq) {
            const int c = q * V;
            float mn[V], mx[V];
            int cmn[V], cmx[V];
            ldv<V>(mn, st + 3 * F + c);
            ldv<V>(mx, st + 4 * F + c);
#pragma unroll
            for (int i = 0; i < V; ++i) { cmn[i] = 0; cmx[i] = 0; }
            for (int t = m.g; t < T; t += m.groups) {
                const int w = frame_weight_fast(t, T, p.f.win_len, p.f.shift_len, inv_shift, n_win, whole);
                if (w == 0) continue;
                float x[V];
                ldv<V>(x, p.f.feat + (f0 + t) * F + c);
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    cmn[i] += x[i] == mn[i] ? w : 0;
                    cmx[i] += x[i] == mx[i] ? w : 0;
                }
            }
            if (m.groups == 1) {
                int32_t* o = p.utt_ties + (long long)u * 2 * F + c;
#pragma unroll
                for (int i = 0; i < V; ++i) { o[i] = cmn[i]; o[F + i] = cmx[i]; }
            } else {
#pragma unroll
                for (int i = 0; i < V; ++i) { sh[0][m.g * F + c + i] = cmn[i]; sh[1][m.g * F + c + i] = cmx[i]; }
            }
        }
    }
    if (m.groups > 1) {
        __syncthreads();
        if (threadIdx.x < m.cols) {
            const int c = threadIdx.x * V;
            int32_t* o = p.utt_ties + (long long)u * 2 * F + c;
#pragma unroll
            for (int i = 0; i < V; ++i) {
                int r1 = 0, r2 = 0;
                for (int k = 0; k < m.groups; ++k) { r1 += sh[0][k * F + c + i]; r2 += sh[1][k * F + c + i]; }
                o[i] = r1; o[F + i] = r2;
            }
        }
    }
}

// Statistics pass 2: one CTA per speaker sums its utterances' tie weights.
__global__ void __launch_bounds__(128 * kBwdMergeSlices) stats_bwd_tie_merge_kernel(const SpeakerStatsBwdParams p) {
    __shared__ int sh[kBwdMergeSlices][2][128];
    const int s = blockIdx.x, F = p.f.n_feat;
    for (int fbase = 0; fbase < F; fbase += 128) {
        const int f = fbase + (threadIdx.x & 127);
        int r0, r1;
        speaker_sum2<int>(p.utt_ties, p.f.spk_ptr, p.f.spk_utts, s, F, f, sh, r0, r1);
        if (threadIdx.x < 128 && f < F) {
            p.spk_ties[(long long)s * 2 * F + f] = r0;
            p.spk_ties[(long long)s * 2 * F + F + f] = r1;
        }
    }
}

// Statistics pass 3: one CTA per utterance writes dfeat from (d mean, d std, d min, d max) of its speaker.
template <int V>
__global__ void __launch_bounds__(kBwdThreads) stats_bwd_frames_kernel(const SpeakerStatsBwdParams p) {
    const int F = p.f.n_feat, u = blockIdx.x;
    const RowMap m(F, V);
    if (!m.active()) return;
    const long long f0 = p.f.frame_off[u];
    const int T = (int)(p.f.frame_off[u + 1] - f0);
    const bool whole = p.f.whole ? p.f.whole[u] != 0 : false;
    const float inv_shift = 1.0f / (float)p.f.shift_len;
    const int n_win = T >= p.f.win_len ? (T - p.f.win_len) / p.f.shift_len + 1 : 0;
    const int s = p.spk_of_utt[u];
    const float* st = p.f.stats + (long long)s * kStatRows * F;
    const float* ds = p.dstats + (long long)s * kStatRows * F;
    const int32_t* ties = p.spk_ties + (long long)s * 2 * F;
    for (int q = m.q0; q < m.cols; q += m.dq) {
        const int c = q * V;
        float mean[V], mn[V], mx[V], cm[V], cs[V], cmn[V], cmx[V];
#pragma unroll
        for (int i = 0; i < V; ++i) {
            const float n = st[c + i], sd = st[2 * F + c + i];
            mean[i] = st[F + c + i]; mn[i] = st[3 * F + c + i]; mx[i] = st[4 * F + c + i];
            cm[i] = ds[F + c + i] / n;
            cs[i] = sd > 0.f ? ds[2 * F + c + i] / (n * sd) : 0.f;      // sigma = 0: no gradient through the std
            cmn[i] = ds[3 * F + c + i] / (float)ties[c + i];
            cmx[i] = ds[4 * F + c + i] / (float)ties[F + c + i];
        }
        for (int t = m.g; t < T; t += m.groups) {
            const int w = frame_weight_fast(t, T, p.f.win_len, p.f.shift_len, inv_shift, n_win, whole);
            float d[V];
            if (w == 0) {
#pragma unroll
                for (int i = 0; i < V; ++i) d[i] = 0.f;
            } else {
                float x[V];
                ldv<V>(x, p.f.feat + (f0 + t) * F + c);
#pragma unroll
                for (int i = 0; i < V; ++i) {
                    float v = fmaf(x[i] - mean[i], cs[i], cm[i]);
                    if (x[i] == mn[i]) v += cmn[i];
                    if (x[i] == mx[i]) v += cmx[i];
                    d[i] = (float)w * v;
                }
            }
            stv<V>(p.dfeat + (f0 + t) * F + c, d);
        }
    }
}

static bool aligned(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

cudaError_t launch_normalize_bwd(const NormalizeBwdParams& p, cudaStream_t stream) {
    if (p.f.n_utts > 0) {
        const bool vec = p.f.n_feat % 4 == 0 && aligned(p.f.feat) && aligned(p.f.stats) && aligned(p.grad) &&
                         (!p.dfeat || aligned(p.dfeat));
        if (vec) normalize_bwd_kernel<4><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
        else normalize_bwd_kernel<1><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
    }
    if (p.dstats && p.n_spk > 0) normalize_bwd_merge_kernel<<<p.n_spk, 128 * kBwdMergeSlices, 0, stream>>>(p);
    return cudaGetLastError();
}

// Both halves pick the vector width from the pointers they touch (the frames half also writes dfeat); the tie weights
// are exact integers, so the width does not change a bit of either result.
static bool stats_bwd_vec(const SpeakerStatsBwdParams& p) {
    return p.f.n_feat % 4 == 0 && aligned(p.f.feat) && aligned(p.f.stats) && (!p.dfeat || aligned(p.dfeat));
}

cudaError_t launch_speaker_stats_bwd_ties(const SpeakerStatsBwdParams& p, cudaStream_t stream) {
    if (p.f.n_utts > 0) {
        if (stats_bwd_vec(p)) stats_bwd_ties_kernel<4><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
        else stats_bwd_ties_kernel<1><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
    }
    if (p.f.n_spk > 0) stats_bwd_tie_merge_kernel<<<p.f.n_spk, 128 * kBwdMergeSlices, 0, stream>>>(p);
    return cudaGetLastError();
}

cudaError_t launch_speaker_stats_bwd_frames(const SpeakerStatsBwdParams& p, cudaStream_t stream) {
    if (p.f.n_utts > 0) {
        if (stats_bwd_vec(p)) stats_bwd_frames_kernel<4><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
        else stats_bwd_frames_kernel<1><<<p.f.n_utts, kBwdThreads, 0, stream>>>(p);
    }
    return cudaGetLastError();
}

}  // namespace sept
