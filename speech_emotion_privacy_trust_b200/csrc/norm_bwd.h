// Launch parameters of the normalisation / statistics backward kernels (norm_bwd.cu).  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>

#include "norm.h"

namespace sept {

struct NormalizeBwdParams {
    // the forward's parameters: feat, frame_off, spk_of_utt, stats, n_feat, mode, n_utts, win_t0, win_len, n_windows
    // (out unused).  win_utt == nullptr selects the frame mode, as in the forward.
    NormalizeParams f;
    const float* grad;           // window mode (n_windows, win_len, F); frame mode (total_frames, F)
    const int32_t* utt_win_ptr;  // window mode: [n_utts + 1] CSR over utt_win
    const int32_t* utt_win;      // window ids of each utterance, sorted by (win_t0, window id)
    float* dfeat;                // (total_frames, F) or null: d/d feat of sum(grad * out)
    // statistics gradient (all null: skipped)
    float* upart;                // workspace (n_utts, 2, F): per utterance S1 = sum gz, S2 = sum gz * z
    const int32_t* spk_ptr;      // [n_spk + 1] CSR over spk_utts
    const int32_t* spk_utts;     // utterance ids grouped by speaker
    int n_spk;
    float* dstats;               // (n_spk, 5, F): 0, d mean, d std, d min, d max
};

struct SpeakerStatsBwdParams {
    SpeakerStatsParams f;        // the forward's parameters (utt_partial unused); stats holds the forward's result
    const int32_t* spk_of_utt;   // [n_utts]
    const float* dstats;         // (n_spk, 5, F); row 0 (count) is ignored
    int32_t* utt_ties;           // workspace (n_utts, 2, F): tie weight of the speaker's min / max in the utterance
    int32_t* spk_ties;           // (n_spk, 2, F), the caller's: written by the ties half, read by the frames half
    float* dfeat;                // (total_frames, F)
};

// workspace of the normalisation backward: the per-utterance (S1, S2) partials
inline size_t normalize_bwd_workspace_bytes(int n_utts, int n_feat) { return (size_t)n_utts * 2 * n_feat * sizeof(float); }

// workspace of the statistics backward's ties half: the utterance tie weights, rounded up to 16 bytes
inline size_t speaker_stats_bwd_ties_workspace_bytes(int n_utts, int n_feat) {
    return ((size_t)n_utts * 2 * n_feat * sizeof(int32_t) + 15) & ~(size_t)15;
}

cudaError_t launch_normalize_bwd(const NormalizeBwdParams& p, cudaStream_t stream);
// the statistics backward in two halves, so that data-parallel callers can sum spk_ties over the ranks in between:
// ties (passes 1 and 2: utt_ties -> spk_ties; dstats and dfeat unused) and frames (pass 3: spk_ties -> dfeat)
cudaError_t launch_speaker_stats_bwd_ties(const SpeakerStatsBwdParams& p, cudaStream_t stream);
cudaError_t launch_speaker_stats_bwd_frames(const SpeakerStatsBwdParams& p, cudaStream_t stream);

}  // namespace sept
