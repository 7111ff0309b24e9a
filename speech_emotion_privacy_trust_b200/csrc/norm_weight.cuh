// Training-window multiplicity of a frame (preprocess_adversary_data.py:26-27, 44-48): the weight of the per-speaker
// statistics, shared by the forward kernels (norm.cu) and their backward (norm_bwd.cu).  Internal header.
#pragma once

namespace sept {

// floor(a / d) for 0 <= a < 2^22 through a float reciprocal (inv = 1.0f / d) and one correction step: exact, and a
// handful of instructions where the integer division costs ~20 -- the statistics kernel was issue bound on it
__device__ __forceinline__ int div_floor_small(int a, int d, float inv) {
    int q = (int)((float)a * inv);
    const int r = a - q * d;
    if (r >= d) ++q;
    else if (r < 0) --q;
    return q;
}

// the same weight with the divisions by `shift` done by div_floor_small; n_win = (T - win) / shift + 1 is passed in
__device__ __forceinline__ int frame_weight_fast(int t, int T, int win, int shift, float inv_shift, int n_win, bool whole) {
    if (whole || T < win) return 1;
    int i_hi = div_floor_small(t, shift, inv_shift);
    if (i_hi > n_win - 1) i_hi = n_win - 1;
    const int num = t - win + 1;
    const int i_lo = num <= 0 ? 0 : div_floor_small(num + shift - 1, shift, inv_shift);
    return i_hi >= i_lo ? i_hi - i_lo + 1 : 0;
}

// number of training windows (start i*shift, length win) that contain frame t of a T-frame utterance (:44-48)
__device__ __forceinline__ int frame_weight(int t, int T, int win, int shift, bool whole) {
    if (whole || T < win) return 1;
    const int n_win = (T - win) / shift + 1;
    int i_hi = t / shift;
    if (i_hi > n_win - 1) i_hi = n_win - 1;
    const int num = t - win + 1;
    const int i_lo = num <= 0 ? 0 : (num + shift - 1) / shift;
    return i_hi >= i_lo ? i_hi - i_lo + 1 : 0;
}

}  // namespace sept
