// Waveform gradient of the MFCC blocks (sm_100a): d(sum Gbar * mfcc) / d wav.  Maths and per-element functions in
// mfcc_bwd.cuh.  The C-ABI layer first recomputes the mel power of both streams with the forward's own launch, then:
//
//   mfcc_bwd_head_kernel          32 frames per CTA, thread = band: stages Gbar of the frames (120 rows, T apart) through
//                                 shared memory with coalesced loads, DCT adjoint of the three streams (the thread's
//                                 basis row in registers), floor routing, stream fold; writes G_0, G_1 over the power,
//                                 per-frame sums of what each stream sends to its floor and per-frame argmax bitmasks
//   mfcc_bwd_route_kernel         one warp per utterance: adds the per-frame sums in frame order and the argmax counts,
//                                 then adds R_s / count at the argmax positions
//   logmel_bwd_frames_kernel<8, 0>  (extract_bwd.cu) the waveform stream on G_0
//   logmel_bwd_frames_kernel<8, 1>  the same frame pass on np.gradient(x) and G_1
//   mfcc_bwd_gather_kernel        one thread per sample: stream 0's rows at the sample plus the np.gradient adjoint of
//                                 stream 1's per-sample sums, recomputed at the neighbours; each sample written once
//
// No atomics anywhere: the result is bit-deterministic and an utterance's gradient does not depend on the batch.
#include <cuda_runtime.h>
#include <cstdint>

#include "mfcc_bwd.cuh"
#include "mfcc_bwd.h"

namespace sept {

namespace {

constexpr int kHeadFrames = 32, kHeadThreads = kMfccBands;
constexpr int kRouteWarps = 4;

__global__ void __launch_bounds__(kHeadThreads) mfcc_bwd_head_kernel(const MfccBwdParams prm) {
    __shared__ float gs[kMfccRows][kHeadFrames];             // Gbar of the CTA's frames: row r, frame f
    __shared__ MfccFloors fl[kHeadFrames];
    __shared__ int mx[2][kHeadFrames];                       // bits of the utterance maxima, streams 0 and 1
    __shared__ float part[3][kHeadThreads / 32][kHeadFrames];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, b = tid;
    const long long TF = prm.total_frames, g0 = (long long)blockIdx.x * kHeadFrames;
    const int nf = TF - g0 < kHeadFrames ? (int)(TF - g0) : kHeadFrames;

    // every warp needs the utterance of the lane's frame for the Gbar loads; warp 0 also keeps its floors and maxima
    const bool live = lane < nf;
    const int u = live ? __ldg(prm.frame_utt + g0 + lane) : 0;
    const long long f0 = live ? __ldg(prm.frames.f.frame_off + u) : 0;
    const long long T = live ? __ldg(prm.frames.f.frame_off + u + 1) - f0 : 0;
    if (warp == 0 && live) {
        const int b0 = __ldg(prm.utt_max + u), b1 = __ldg(prm.utt_max + prm.frames.f.n_utts + u);
        mx[0][lane] = b0;
        mx[1][lane] = b1;
        fl[lane] = mfcc_floors(__int_as_float(b0), __int_as_float(b1));
    }
    // lanes = consecutive frames (consecutive addresses inside an utterance), warps = rows
    const float* src = prm.grad + f0 * kMfccRows + (g0 + lane - f0);
    for (int r = warp; r < kMfccRows; r += kHeadThreads / 32) gs[r][lane] = live ? __ldg(src + r * T) : 0.f;

    float d[kMfccCoefs];                                     // basis row of the thread's band
#pragma unroll
    for (int i = 0; i < kMfccCoefs / 4; ++i) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(prm.dct + b * kMfccCoefs) + i);
        d[4 * i] = q.x; d[4 * i + 1] = q.y; d[4 * i + 2] = q.z; d[4 * i + 3] = q.w;
    }
    __syncthreads();

    float* pw0 = prm.power + g0 * kMfccBands + b;
    float* pw1 = pw0 + TF * kMfccBands;
#pragma unroll 2
    for (int f = 0; f < nf; ++f) {
        const float p0 = pw0[f * kMfccBands], p1 = pw1[f * kMfccBands];
        const MfccHead h = mfcc_head_one([&](int r) { return gs[r][f]; }, d, p0, p1, fl[f]);
        pw0[f * kMfccBands] = h.g0;                          // in place: this thread's own power values, already read
        pw1[f * kMfccBands] = h.g1;
        const unsigned m0 = __ballot_sync(0xffffffffu, __float_as_int(p0) == mx[0][f]);
        const unsigned m1 = __ballot_sync(0xffffffffu, __float_as_int(p1) == mx[1][f]);
        float r0 = h.r[0], r1 = h.r[1], r2 = h.r[2];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            r0 += __shfl_xor_sync(0xffffffffu, r0, o);
            r1 += __shfl_xor_sync(0xffffffffu, r1, o);
            r2 += __shfl_xor_sync(0xffffffffu, r2, o);
        }
        if (lane == 0) {
            part[0][warp][f] = r0;
            part[1][warp][f] = r1;
            part[2][warp][f] = r2;
            uint32_t* am = prm.amask + (g0 + f) * 8;
            am[warp] = m0;
            am[4 + warp] = m1;
        }
    }
    __syncthreads();
    if (tid < nf) {
        float4 o;
        o.x = ((part[0][0][tid] + part[0][1][tid]) + part[0][2][tid]) + part[0][3][tid];
        o.y = ((part[1][0][tid] + part[1][1][tid]) + part[1][2][tid]) + part[1][3][tid];
        o.z = ((part[2][0][tid] + part[2][1][tid]) + part[2][2][tid]) + part[2][3][tid];
        o.w = 0.f;
        reinterpret_cast<float4*>(prm.part)[g0 + tid] = o;
    }
}

__global__ void __launch_bounds__(kRouteWarps * 32) mfcc_bwd_route_kernel(const MfccBwdParams prm) {
    const int lane = threadIdx.x & 31, u = blockIdx.x * kRouteWarps + (threadIdx.x >> 5);
    if (u >= prm.frames.f.n_utts) return;
    const long long f0 = __ldg(prm.frames.f.frame_off + u), f1 = __ldg(prm.frames.f.frame_off + u + 1);
    float r0 = 0.f, r1 = 0.f, r2 = 0.f;
    int c0 = 0, c1 = 0;
    for (long long f = f0 + lane; f < f1; f += 32) {
        const float4 p = __ldg(reinterpret_cast<const float4*>(prm.part) + f);
        r0 += p.x; r1 += p.y; r2 += p.z;
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(prm.amask) + 2 * f);
        const uint4 c = __ldg(reinterpret_cast<const uint4*>(prm.amask) + 2 * f + 1);
        c0 += __popc(a.x) + __popc(a.y) + __popc(a.z) + __popc(a.w);
        c1 += __popc(c.x) + __popc(c.y) + __popc(c.z) + __popc(c.w);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        r0 += __shfl_xor_sync(0xffffffffu, r0, o);
        r1 += __shfl_xor_sync(0xffffffffu, r1, o);
        r2 += __shfl_xor_sync(0xffffffffu, r2, o);
        c0 += __shfl_xor_sync(0xffffffffu, c0, o);
        c1 += __shfl_xor_sync(0xffffffffu, c1, o);
    }
    const float s0 = c0 ? r0 / (float)c0 : 0.f, s1 = c1 ? r1 / (float)c1 : 0.f, s2 = c1 ? r2 / (float)c1 : 0.f;
    if (s0 == 0.f && s1 == 0.f && s2 == 0.f) return;        // nothing was floored (the usual case: no write at all)
    const float max1 = __int_as_float(__ldg(prm.utt_max + prm.frames.f.n_utts + u));
    float* G0 = prm.power;
    float* G1 = prm.power + prm.total_frames * kMfccBands;
    for (long long f = f0 + lane; f < f1; f += 32) {
        for (int w = 0; w < 8; ++w) {
            for (unsigned bits = prm.amask[f * 8 + w]; bits; bits &= bits - 1) {
                const long long i = f * kMfccBands + (w & 3) * 32 + (__ffs(bits) - 1);
                if (w < 4) mfcc_add_share0(G0[i], s0);
                else mfcc_add_share1(G1[i], s1, s2, max1);
            }
        }
    }
}

__global__ void __launch_bounds__(256) mfcc_bwd_gather_kernel(const MfccBwdParams prm) {
    const ExtractParams& fp = prm.frames.f;
    const int row = Bwd<Geo<8>>::row_floats(200);
    const long long first = __ldg(fp.utt_off), last = __ldg(fp.utt_off + fp.n_utts);
    for (long long i = first + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < last; i += (long long)gridDim.x * blockDim.x) {
        const int u = find_utt(fp.utt_off, fp.n_utts, i);
        const long long s0 = __ldg(fp.utt_off + u);
        const int n = (int)(__ldg(fp.utt_off + u + 1) - s0);
        const int i0 = __ldg(fp.item_off + u), n_items = __ldg(fp.item_off + u + 1) - i0;
        prm.dwav[i] = mfcc_bwd_gather(prm.rows0 + (long long)i0 * row, prm.rows1 + (long long)i0 * row, row, n_items, n,
                                      (int)(i - s0));
    }
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

}  // namespace

MfccBwdLayout mfcc_bwd_layout(int n_utts, long long total_frames, long long n_items) {
    MfccBwdLayout l{};
    if (n_utts <= 0 || total_frames <= 0 || n_items <= 0) return l;
    const size_t tf = (size_t)total_frames, row = (size_t)Bwd<Geo<8>>::row_floats(200);
    size_t o = 0;
    l.power = o;     o = align256(o + 2 * tf * kMfccBands * sizeof(float));
    l.frame_utt = o; o = align256(o + tf * sizeof(int32_t));
    l.utt_max = o;   o = align256(o + 2 * (size_t)n_utts * sizeof(int32_t));
    l.part = o;      o = align256(o + tf * 4 * sizeof(float));
    l.amask = o;     o = align256(o + tf * 8 * sizeof(uint32_t));
    l.rows0 = o;     o = align256(o + (size_t)n_items * row * sizeof(float));
    l.rows1 = o;     o = align256(o + (size_t)n_items * row * sizeof(float));
    l.bytes = o;
    return l;
}

cudaError_t launch_mfcc_bwd(const MfccBwdParams& prm, int sms, cudaStream_t stream) {
    const long long head_blocks = (prm.total_frames + kHeadFrames - 1) / kHeadFrames;
    mfcc_bwd_head_kernel<<<(unsigned)head_blocks, kHeadThreads, 0, stream>>>(prm);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    mfcc_bwd_route_kernel<<<(prm.frames.f.n_utts + kRouteWarps - 1) / kRouteWarps, kRouteWarps * 32, 0, stream>>>(prm);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    LogmelBwdParams fp = prm.frames;
    fp.grad = prm.power;
    fp.ws = prm.rows0;
    if ((e = launch_logmel_bwd_frames_400(fp, 0, sms, stream)) != cudaSuccess) return e;
    fp.grad = prm.power + prm.total_frames * kMfccBands;
    fp.ws = prm.rows1;
    if ((e = launch_logmel_bwd_frames_400(fp, 1, sms, stream)) != cudaSuccess) return e;
    mfcc_bwd_gather_kernel<<<sms * 8, 256, 0, stream>>>(prm);
    return cudaGetLastError();
}

}  // namespace sept
