// Launch parameters of the waveform-domain cloak kernels (wave_cloak.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace sept {

constexpr int kWaveThreads = 256;     // threads per CTA of every kernel; also the tiles staged per chunk
constexpr int kWaveSlices = 592;      // backward: partial rows (4 per B200 SM).  A constant, not the SM count: the
                                      // summation order, and so the bits of the gradient, are the same on every GPU
constexpr int kWaveMergeLanes = 8;    // backward: lanes of the ordered slice sum (kWaveSlices / 8 = 74 slices each)

struct WaveAddParams {
    const float* x;          // (n) 16-byte aligned
    const int64_t* utt_off;  // (n_utts + 1) device
    int n_utts;
    int64_t n;
    const float* noise;      // (period) 16-byte aligned
    int period;              // multiple of 4
    float* y;                // (n) 16-byte aligned
};

struct WaveReduceParams {
    const float* g;          // (n) 16-byte aligned
    const int64_t* utt_off;  // (n_utts + 1) device
    const int64_t* tile_off; // (n_utts + 1) device: tiles of utterance u are tile_off[u] .. tile_off[u+1]-1
    int n_utts;
    int64_t n_tiles;         // tile_off[n_utts]
    int period;              // multiple of 4
    float* partial;          // workspace (kWaveSlices, period)
    float* r;                // (period)
};

struct WaveEvalParams {
    const float* x;          // (n) 16-byte aligned
    const int64_t* utt_off;  // (n_utts + 1) device
    int n_utts;
    int64_t n;
    const float* locs;       // (period) 16-byte aligned
    const float* rhos;       // (period) 16-byte aligned
    const float* eps;        // (n_utts, period) 16-byte aligned, or null -> Philox(seed, offset)
    uint64_t seed, offset;
    const uint64_t* draw;    // device counter or null (0)
    const int64_t* utt_draw; // (n_utts) device draw index of each utterance, or null (u)
    float eps_std, min_scale, max_scale;
    int period;              // multiple of 4
    float* sigma;            // workspace (period): sigma(rhos), written by the pre-pass
    float* y;                // (n) 16-byte aligned
};

struct WaveReducePerUttParams {
    WaveReduceParams r;      // partial: workspace (2, kWaveSlices, period), the rows of g then those of g * eps_u; r: dlocs
    const float* rhos;       // (period) 16-byte aligned
    const float* eps;        // (n_utts, period) 16-byte aligned, or null -> Philox(seed, offset), as in WaveEvalParams
    uint64_t seed, offset;
    const uint64_t* draw;    // device draw base or null (0)
    const int64_t* utt_draw; // (n_utts) device draw index of each utterance, or null (u)
    float eps_std, min_scale, max_scale;
    float* drhos;            // (period) 16-byte aligned
};

cudaError_t launch_wave_add(const WaveAddParams& p, cudaStream_t stream);
cudaError_t launch_wave_eval(const WaveEvalParams& p, cudaStream_t stream);
cudaError_t launch_wave_reduce(const WaveReduceParams& p, cudaStream_t stream);
cudaError_t launch_wave_reduce_per_utt(const WaveReducePerUttParams& p, cudaStream_t stream);

}  // namespace sept
