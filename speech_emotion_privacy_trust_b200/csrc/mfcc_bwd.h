// Launch parameters and workspace layout of the MFCC backward (mfcc_bwd.cu), shared with the C-ABI layer (api.cu).
// Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

#include "extract_bwd.h"

namespace sept {

// Byte offsets into the workspace (each 256-byte aligned).  The recomputed mel power of both streams is overwritten in
// place by the head kernel with the dB gradients G_0, G_1 of the two frame passes.
struct MfccBwdLayout {
    size_t power;        // float [2][total_frames][128]: mel power of x and of np.gradient(x); then G_0, G_1
    size_t frame_utt;    // int32 [total_frames]: utterance of each frame (written by the power kernel)
    size_t utt_max;      // int32 [2][n_utts]: bits of the largest mel power per utterance and stream
    size_t part;         // float [total_frames][4]: per-frame sums of what streams 0, 1, 2 send to their floor
    size_t amask;        // uint32 [total_frames][8]: argmax bands per frame, stream 0 (words 0-3) and 1 (words 4-7)
    size_t rows0, rows1; // float [n_items][row]: span rows of the two frame passes
    size_t bytes;
};
MfccBwdLayout mfcc_bwd_layout(int n_utts, long long total_frames, long long n_items);

struct MfccBwdParams {
    LogmelBwdParams frames;      // wav, offsets, n_fft 400 constants and n_items of both frame passes (grad, ws per pass)
    const float* grad;           // (120, T_u) blocks of sept_mfcc_f32's layout
    const float* dct;            // [128][40] orthonormal DCT-II basis
    const int32_t* frame_utt;
    const int32_t* utt_max;
    long long total_frames;
    float* power;                // [2][total_frames][128] in: mel power; out: G_0, G_1
    float* part;
    uint32_t* amask;
    float* rows0;
    float* rows1;
    float* dwav;
};

// head, route, the two frame passes, gather; the power must already be in prm.power (the forward's power launch)
cudaError_t launch_mfcc_bwd(const MfccBwdParams& prm, int sms, cudaStream_t stream);

}  // namespace sept
