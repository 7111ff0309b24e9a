// Launch parameters of the polyphase sinc resampler (resample.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>

namespace sept {

struct ResampleParams {
    const float* in;            // ragged input, all utterances back to back
    const int64_t* in_off;      // [n_utts + 1]
    const int64_t* out_off;     // [n_utts + 1], any length per utterance; sept_resample_layout gives torchaudio's
    int n_utts;
    int orig, up;               // orig_freq / gcd, new_freq / gcd
    int width;                  // zero-crossing half width in input samples (torchaudio's `width`)
    int taps;                   // stored taps per phase
    const int32_t* k_lo;        // [up] first stored tap of each phase (index into the torchaudio kernel row)
    const float* w;             // [up][taps] kernel rows restricted to their non-zero support
    float* out;
    long long total_out;
    // register-tile tables (tables.h: make_resample_tiles); tile_wt null: only the one-thread-per-sample kernel is available
    const int32_t* tile_base;   // [n_groups]
    const float* tile_wt;       // [n_groups][tg][4]
    int n_groups, tg, base_min, base_max;
};

cudaError_t launch_resample(const ResampleParams& p, cudaStream_t stream);
cudaError_t launch_pcm16_to_f32(const short* in, long long n, float* out, cudaStream_t stream);

}  // namespace sept
