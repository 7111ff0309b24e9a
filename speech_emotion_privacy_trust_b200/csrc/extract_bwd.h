// Launch parameters of the log-mel backward (extract_bwd.cu), shared with the C-ABI layer (api.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

#include "extract.h"

namespace sept {

struct LogmelBwdParams {
    ExtractParams f;             // the forward's launch, which the frame pass recomputes (its outputs are unused)
    long long n_items;           // items the workspace holds rows for
    const float* grad;           // (total_frames, n_mels) upstream gradient of the frame-major log-mel
    float* ws;                   // [n_items][row] span rows
    float* dwav;                 // gradient w.r.t. wav
};

size_t logmel_bwd_workspace_bytes(int n_fft, int hop, long long n_items);
cudaError_t launch_logmel_bwd(const LogmelBwdParams& prm, int n_fft, int sms, cudaStream_t stream);

// The frame pass alone at n_fft 400 (rows to prm.ws, no gather).  deriv: stage np.gradient(x) instead of x.
cudaError_t launch_logmel_bwd_frames_400(const LogmelBwdParams& prm, int deriv, int sms, cudaStream_t stream);

}  // namespace sept
