// Launch parameters of the log-mel backward (extract_bwd.cu), shared with the C-ABI layer (api.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

namespace sept {

struct LogmelBwdParams {
    const float* wav;            // all utterances back to back
    const int64_t* utt_off;      // [n_utts + 1] sample offsets
    const int64_t* frame_off;    // [n_utts + 1] frame offsets
    const int32_t* item_off;     // [n_utts + 1] item offsets
    int n_utts;
    long long n_items;           // items the workspace holds rows for
    int hop;
    int n_mels;
    int n_mel_entries, n_mel_head;
    int fast_dn;                 // the forward runs its compiled-in 128-band path: falling weight = 1/4 - rising
    const float* window;         // [n_fft] periodic Hann
    const float* tws;            // split twiddles (tables.h: make_split_twiddles)
    const void* mel_prog;        // gather program (tables.h: make_mel_program)
    const float* grad;           // (total_frames, n_mels) upstream gradient of the frame-major log-mel
    float* ws;                   // [n_items][row] span rows
    float* dwav;                 // gradient w.r.t. wav
};

size_t logmel_bwd_workspace_bytes(int n_fft, int hop, long long n_items);
cudaError_t launch_logmel_bwd(const LogmelBwdParams& prm, int n_fft, int sms, cudaStream_t stream);

// The frame pass alone at n_fft 400 (rows to prm.ws, no gather).  deriv: stage np.gradient(x) instead of x.
cudaError_t launch_logmel_bwd_frames_400(const LogmelBwdParams& prm, int deriv, int sms, cudaStream_t stream);

}  // namespace sept
