// Waveform gradient of the frame-major log-mel (sm_100a): d(sum G * logmel) / d wav.  Maths and per-lane phases in
// extract_bwd.cuh.
//
//   logmel_bwd_frames_kernel<R, DERIV>  persistent, one CTA per SM, one warp per item: recompute spectrum, power and mel
//                                power with the forward's phase functions, form dM and dP, inverse split, inverse
//                                prime-factor transform, window, overlap-add of the item's frames -> one workspace row per
//                                item.  DERIV = 1 stages np.gradient(x) instead of x (the MFCC backward, mfcc_bwd.cu).
//   logmel_bwd_gather_kernel<R>  one thread per waveform sample: sums the rows covering it (and its reflect mirrors) in
//                                item order and writes dwav once.  No atomics: the result is bit-deterministic and an
//                                utterance's gradient does not depend on the rest of the batch.
#include <cuda_runtime.h>
#include <cstdint>

#include "extract_bwd.cuh"
#include "extract_bwd.h"

namespace sept {

template <int R, int DERIV = 0>
__global__ void __launch_bounds__(kBwdWarps * 32, 1) logmel_bwd_frames_kernel(const LogmelBwdParams prm) {
    using G = Geo<R>;
    using B = Bwd<G>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
    const int hop = prm.hop, n_mels = prm.n_mels;

    mel_step* melp = reinterpret_cast<mel_step*>(smem_raw);
    f2* win2 = reinterpret_cast<f2*>(melp + prm.n_mel_entries);
    f2* tws = win2 + G::NC;
    for (int i = threadIdx.x; i < 13 * G::TWS; i += blockDim.x) tws[i] = reinterpret_cast<const f2*>(prm.tws)[i];
    for (int i = threadIdx.x; i < prm.n_mel_entries; i += blockDim.x)
        reinterpret_cast<f4*>(melp)[i] = reinterpret_cast<const f4*>(prm.mel_prog)[i];
    for (int i = threadIdx.x; i < G::NC; i += blockDim.x) win2[i] = reinterpret_cast<const f2*>(prm.window)[i];
    __syncthreads();

    float* wbase = reinterpret_cast<float*>(smem_raw + bwd_const_bytes(R, prm.n_mel_entries)) + (size_t)warp * B::warp_floats(hop, n_mels);
    float* stage = wbase;
    pk2* Y = reinterpret_cast<pk2*>(stage + G::stage_floats(hop));
    pk2* P = Y + G::Y_PK2;
    pk2* U = P + G::PPW * G::PP;
    pk2* D = reinterpret_cast<pk2*>(reinterpret_cast<float*>(U) + B::ud_floats(n_mels));
    const mel_step* prog = melp;
    const int row = B::row_floats(hop), span = G::span(hop);

    long long n_items = __ldg(prm.item_off + prm.n_utts);
    if (n_items > prm.n_items) n_items = prm.n_items;
    for (long long item = (long long)blockIdx.x * warps + warp; item < n_items; item += (long long)gridDim.x * warps) {
        const int u = bwd_find_utt(prm.item_off, prm.n_utts, item);
        const long long s0 = __ldg(prm.utt_off + u), f0 = __ldg(prm.frame_off + u);
        const int n = (int)(__ldg(prm.utt_off + u + 1) - s0);
        const int T = (int)(__ldg(prm.frame_off + u + 1) - f0);
        const int t0 = (int)(item - __ldg(prm.item_off + u)) * G::FPW;
        __syncwarp();                                            // previous item's frame tile reads are done
        stage_item<G>(lane, prm.wav + s0, n, t0, hop, DERIV, stage);
        __syncwarp();
        pass1<G, false>(lane, stage, hop, WinShared{win2}, Y);
        __syncwarp();
#pragma unroll 1
        for (int task = lane; task < G::P2_TASKS; task += 32) pass2_row<G>(task, Y);
        __syncwarp();
        bwd_row0_copy<G>(lane, Y);
        __syncwarp();
        bwd_split<G>(lane, Y, tws, P);
        __syncwarp();
        bwd_mel_sums<G>(lane, P, prog, prm.n_mel_head, n_mels, prm.fast_dn != 0, U, D);
        __syncwarp();
        bwd_dmel<G>(lane, U, D, prm.grad + f0 * n_mels, T, t0, n_mels, P);
        __syncwarp();
        bwd_dpower<G>(lane, U, prog, prm.n_mel_head, n_mels, P);
        __syncwarp();
        bwd_unsplit<G>(lane, Y, P, tws);
        __syncwarp();
#pragma unroll 1
        for (int task = lane; task < G::P2_TASKS; task += 32) pass2_row<G>(task, Y);
        __syncwarp();
        {
            pk2 gr[25], gi[25];
            bwd_pass1_load<G>(lane, Y, win2, gr, gi);
            __syncwarp();
            bwd_pass1_store<G>(lane, reinterpret_cast<float*>(Y), gr, gi);
        }
        __syncwarp();
        float* out = prm.ws + item * row;
        for (int j = lane; j < span; j += 32) out[j] = bwd_ola<G>(j, reinterpret_cast<const float*>(Y), hop);
    }
}

template <int R>
__global__ void __launch_bounds__(256) logmel_bwd_gather_kernel(const LogmelBwdParams prm) {
    using G = Geo<R>;
    const int row = Bwd<G>::row_floats(prm.hop);
    const long long first = __ldg(prm.utt_off), last = __ldg(prm.utt_off + prm.n_utts);
    for (long long i = first + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < last; i += (long long)gridDim.x * blockDim.x) {
        const int u = bwd_find_utt(prm.utt_off, prm.n_utts, i);
        const long long s0 = __ldg(prm.utt_off + u);
        const int n = (int)(__ldg(prm.utt_off + u + 1) - s0);
        const int i0 = __ldg(prm.item_off + u), n_items = __ldg(prm.item_off + u + 1) - i0;
        prm.dwav[i] = bwd_gather<G>(prm.ws + (long long)i0 * row, row, n_items, n, (int)(i - s0), prm.hop);
    }
}

constexpr size_t kBwdMaxSmem = 232448;

template <int R>
static int bwd_warps(int hop, int n_mels, int n_mel_entries) {
    const size_t cb = (size_t)bwd_const_bytes(R, n_mel_entries), wb = (size_t)Bwd<Geo<R>>::warp_floats(hop, n_mels) * 4;
    if (cb + wb > kBwdMaxSmem) return 0;
    const int fit = (int)((kBwdMaxSmem - cb) / wb);
    return fit < kBwdWarps ? fit : kBwdWarps;
}

template <int R, int DERIV>
static cudaError_t launch_frames(const LogmelBwdParams& prm, int sms, cudaStream_t stream) {
    const auto kernel = logmel_bwd_frames_kernel<R, DERIV>;
    const int warps = bwd_warps<R>(prm.hop, prm.n_mels, prm.n_mel_entries);
    if (warps == 0) return cudaErrorInvalidConfiguration;
    const size_t smem = (size_t)bwd_const_bytes(R, prm.n_mel_entries) +
                        (size_t)warps * Bwd<Geo<R>>::warp_floats(prm.hop, prm.n_mels) * 4;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<sms, warps * 32, smem, stream>>>(prm);
    return cudaGetLastError();
}

template <int R>
static cudaError_t launch_r(const LogmelBwdParams& prm, int sms, cudaStream_t stream) {
    cudaError_t e = launch_frames<R, 0>(prm, sms, stream);
    if (e != cudaSuccess) return e;
    logmel_bwd_gather_kernel<R><<<sms * 8, 256, 0, stream>>>(prm);
    return cudaGetLastError();
}

cudaError_t launch_logmel_bwd(const LogmelBwdParams& prm, int n_fft, int sms, cudaStream_t stream) {
    switch (n_fft) {
        case 400: return launch_r<8>(prm, sms, stream);
        case 800: return launch_r<16>(prm, sms, stream);
        case 1600: return launch_r<32>(prm, sms, stream);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_logmel_bwd_frames_400(const LogmelBwdParams& prm, int deriv, int sms, cudaStream_t stream) {
    return deriv ? launch_frames<8, 1>(prm, sms, stream) : launch_frames<8, 0>(prm, sms, stream);
}

size_t logmel_bwd_workspace_bytes(int n_fft, int hop, long long n_items) {
    if (n_items <= 0 || hop <= 0) return 0;
    int row = 0;
    switch (n_fft) {
        case 400: row = Bwd<Geo<8>>::row_floats(hop); break;
        case 800: row = Bwd<Geo<16>>::row_floats(hop); break;
        case 1600: row = Bwd<Geo<32>>::row_floats(hop); break;
        default: return 0;
    }
    return (size_t)n_items * row * sizeof(float);
}

}  // namespace sept
