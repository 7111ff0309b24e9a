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
    const ExtractParams& f = prm.f;
    const int hop = f.hop, n_mels = f.n_mels;

    const CtaConsts cc = load_cta_consts<G>(threadIdx.x, blockDim.x, smem_raw, f);
    const f2* win2 = cc.win2;
    const f2* tws = cc.tws;
    __syncthreads();

    float* wbase = reinterpret_cast<float*>(smem_raw + extract_const_bytes(R, f.n_mel_entries)) + (size_t)warp * B::warp_floats(hop, n_mels);
    float* stage = wbase;
    pk2* Y = reinterpret_cast<pk2*>(stage + G::stage_floats(hop));
    pk2* P = Y + G::Y_PK2;
    pk2* U = P + G::PPW * G::PP;
    pk2* D = reinterpret_cast<pk2*>(reinterpret_cast<float*>(U) + B::ud_floats(n_mels));
    const mel_step* prog = cc.mel;
    const int row = B::row_floats(hop), span = G::span(hop);

    long long n_items = __ldg(f.item_off + f.n_utts);
    if (n_items > prm.n_items) n_items = prm.n_items;
    for (long long item = (long long)blockIdx.x * warps + warp; item < n_items; item += (long long)gridDim.x * warps) {
        const int u = find_utt(f.item_off, f.n_utts, item);
        const long long s0 = __ldg(f.utt_off + u), f0 = __ldg(f.frame_off + u);
        const int n = (int)(__ldg(f.utt_off + u + 1) - s0);
        const int T = (int)(__ldg(f.frame_off + u + 1) - f0);
        const int t0 = (int)(item - __ldg(f.item_off + u)) * G::FPW;
        __syncwarp();                                            // previous item's frame tile reads are done
        stage_item<G>(lane, f.wav + s0, n, t0, hop, DERIV, stage);
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
        bwd_mel_sums<G>(lane, P, prog, f.n_mel_head, n_mels, f.mel_fast != 0, U, D);
        __syncwarp();
        bwd_dmel<G>(lane, U, D, prm.grad + f0 * n_mels, T, t0, n_mels, P);
        __syncwarp();
        bwd_dpower<G>(lane, U, prog, f.n_mel_head, n_mels, P);
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
    const ExtractParams& f = prm.f;
    const int row = Bwd<G>::row_floats(f.hop);
    const long long first = __ldg(f.utt_off), last = __ldg(f.utt_off + f.n_utts);
    for (long long i = first + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < last; i += (long long)gridDim.x * blockDim.x) {
        const int u = find_utt(f.utt_off, f.n_utts, i);
        const long long s0 = __ldg(f.utt_off + u);
        const int n = (int)(__ldg(f.utt_off + u + 1) - s0);
        const int i0 = __ldg(f.item_off + u), n_items = __ldg(f.item_off + u + 1) - i0;
        prm.dwav[i] = bwd_gather<G>(prm.ws + (long long)i0 * row, row, n_items, n, (int)(i - s0), f.hop);
    }
}

template <int R, int DERIV>
static cudaError_t launch_frames(const LogmelBwdParams& prm, int sms, cudaStream_t stream) {
    const auto kernel = logmel_bwd_frames_kernel<R, DERIV>;
    const size_t cb = extract_const_bytes(R, prm.f.n_mel_entries), wb = Bwd<Geo<R>>::warp_floats(prm.f.hop, prm.f.n_mels) * 4;
    const int warps = warps_that_fit(cb, wb, kBwdWarps, kMaxDynSmem);
    if (warps == 0) return cudaErrorInvalidConfiguration;
    const size_t smem = cb + warps * wb;
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
