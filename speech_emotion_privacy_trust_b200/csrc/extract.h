// Launch parameters shared by extract.cu and the C-ABI layer (api.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace sept {

enum : int {
    kModeDbFrameMajor = 0,   // out[(frame_off[u] + t) * n_mels + m]            log-mel dB, (T, n_mels) per utterance
    kModeDbBandMajor = 1,    // out[frame_off[u] * n_mels + m * T_u + t]        log-mel dB, (n_mels, T) per utterance
    kModeMfccPower = 2,      // out[(s * total_frames + frame_off[u] + t) * n_mels + m]  raw mel power of streams
                             // s = 0 (waveform) and s = 1 (np.gradient of it) + per-utterance max into utt_max
};

// warps per CTA (one persistent CTA per SM).  8 warps = 2 per scheduler = 255 registers per thread: the fused pass 2 +
// split keeps two spectrum rows of a frame pair in registers (~200); 11 warps would fit the 227 KB of shared memory but
// leave 168 registers, and the spills cost more than the extra warps give (measured 4.55 ms vs 3.94 ms per step; n_fft 1600
// with ten warps and items drawn from a counter: 7.11 vs 6.95 ms).
template <int R> struct ExtractWarps { static constexpr int value = 8; };

struct ExtractParams {
    const float* wav;            // all utterances back to back
    const int64_t* utt_off;      // [n_utts + 1] sample offsets
    const int64_t* frame_off;    // [n_utts + 1] frame offsets, T_u = 1 + N_u / hop
    const int32_t* item_off;     // [n_utts + 1] item offsets, ceil(T_u / FPW) items per utterance
    int n_utts;
    int hop;
    int n_mels;
    int n_mel_entries;           // 16-byte entries of the mel gather program (head + steps x width)
    int n_mel_head;              // broadcast entries of interval 0 in front of the program
    int mel_fast;                // the program has the compiled-in step counts of the 128-mel filterbank (extract_mel_fast_ok)
    int deriv;                   // dB modes: 0 waveform, 1 np.gradient(waveform)
    long long total_frames;      // kModeMfccPower only
    const float* window;         // [n_fft] periodic Hann
    const float* tws;            // [13][R][4] split twiddles
    const void* mel_prog;        // [n_mel_entries] {float up, dn; int byte offset, pad} (tables.h: make_mel_program)
    float* out;
    int* utt_max;                // kModeMfccPower: [2][n_utts] float bits, zeroed by the caller
    int* frame_utt;              // kModeMfccPower: [total_frames] utterance of every frame
};

struct MfccDctParams {
    const float* power;          // [2][total_frames][128] from kModeMfccPower
    const int* utt_max;          // [2][n_utts]
    const int* frame_utt;        // [total_frames] from kModeMfccPower
    const int64_t* frame_off;    // [n_utts + 1]
    const float* dct;            // [128][40]
    int n_utts;
    long long total_frames;
    float top_db;
    float* out;                  // per utterance (120, T_u) at frame_off[u] * 120
};

cudaError_t launch_extract(const ExtractParams& prm, int n_fft, int mode, int grid, cudaStream_t stream);
size_t extract_smem_bytes_for(int n_fft, int hop, int n_mel_entries);
int extract_frames_per_item(int n_fft);
// true when a 128-band program with these step counts may run the unrolled mel path
bool extract_mel_fast_ok(int n_fft, int n_mels, int n_head, const int* round_steps, int n_rounds);
cudaError_t launch_mfcc_dct(const MfccDctParams& prm, cudaStream_t stream);        // dB + top_db floor + DCT (mfcc_dct.cu)

}  // namespace sept
