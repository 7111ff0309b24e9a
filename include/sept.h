/* sept.h -- C ABI of libsept_b200: B200-native (sm_100a) speech feature extraction + cloak / gradient-reversal path.
 *
 * Drop-in boundary for the hot path of usc-sail/speech-emotion-privacy-trust.  The reference has no FFI (it is pure
 * Python); each entry point below names the reference Python interface it replaces (file:line, relative to the
 * reference tree, or torchaudio/ for the un-vendored third-party code the arithmetic lives in).  INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer named *_dev is DEVICE memory owned by the caller (e.g. a torch tensor's data_ptr); every buffer is
 *     allocated by the caller; the library owns only an immutable per-device cache of constants (Hann window, split
 *     twiddles, mel band weights, DCT basis, resampling rows) created on first use or by sept_init().
 *   - `stream` is a cudaStream_t (pass torch.cuda.current_stream().cuda_stream); calls enqueue work and return; after
 *     sept_init() they neither allocate nor synchronise, so they can be captured into CUDA graphs.
 *   - return value: 0 on success, a negative SEPT_E_* code otherwise; sept_last_error() gives the text (thread local).
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with SEPT_E_CUDA.
 *   - float tensors are fp32, contiguous; float4 paths need 16-byte aligned pointers (torch allocations are).
 */
#ifndef SEPT_H_
#define SEPT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SEPT_OK 0
#define SEPT_E_BADARG (-1)       /* null pointer, negative size, misaligned or inconsistent argument            */
#define SEPT_E_UNSUPPORTED (-2)  /* n_fft not in {400, 800, 1600}, odd hop, n_mels/hop too large for shared memory */
#define SEPT_E_TOO_SHORT (-3)    /* an utterance has <= n_fft/2 samples: reflect padding impossible (torch.stft raises too) */
#define SEPT_E_CUDA (-4)         /* CUDA runtime error, text in sept_last_error()                                */

#define SEPT_LAYOUT_FRAME_MAJOR 0 /* per utterance (T, n_mels): what preprocess_adversary_data.py:345 consumes (mel1[0].T) */
#define SEPT_LAYOUT_BAND_MAJOR 1  /* per utterance (n_mels, T): what mel_spectrogram() returns                   */

#define SEPT_NORM_ZNORM 0
#define SEPT_NORM_MINMAX 1

typedef void* sept_stream_t; /* cudaStream_t */

int sept_version(void);
const char* sept_last_error(void);
/* "SEPT_SRC_HASH=<sha256 of the sources this library was compiled from>": the Python loader refuses (or rebuilds) a
 * library whose hash differs from the sources next to it, so a stale prebuilt .so is never tested silently. */
const char* sept_source_hash(void);

/* Build the constant cache of the current device for n_fft in {400, 800, 1600} x n_mels, and the 128x40 DCT basis.
 * The log-mel backward (sept_logmel_bwd_f32) runs on the same constants.
 * Optional (first use does it), but call it before CUDA-graph capture. */
int sept_init(int n_mels);

/* ---- extraction ------------------------------------------------------------------------------------------------
 * A batch is a ragged concatenation: utterance u is wav[utt_off[u] : utt_off[u+1]].
 * Frames: T_u = 1 + N_u / hop (center=True).  Items: the kernel's work unit, sept_frames_per_item(n_fft) frames.   */

/* frames per work item for this n_fft (8 / 4 / 2 for 400 / 800 / 1600); 0 if unsupported */
int sept_frames_per_item(int n_fft);

/* HOST helper: from host utt_off[n_utts+1] fill host frame_off[n_utts+1] and item_off[n_utts+1]; validates lengths
 * (SEPT_E_TOO_SHORT like torch.stft's reflect-pad check, torch/functional.py:675-680). */
int sept_extract_layout(const int64_t* utt_off_host, int n_utts, int n_fft, int hop, int64_t* frame_off_host,
                        int32_t* item_off_host);

/* log-mel dB of a ragged batch.  Replaces mel_spectrogram(audio, n_fft, feature_len)
 * (feature_extraction/audio_feature_extraction.py:29-46 -> torchaudio/transforms/_transforms.py:566-631, 300-346):
 * reflect pad n_fft/2, frames of n_fft at stride hop, periodic Hann, rFFT, |X|^2, HTK mel (0..8 kHz, norm None),
 * 10*log10(max(., 1e-10)).  deriv=1 extracts from np.gradient(waveform) instead (audio_feature_extraction.py:20).
 * out_dev holds total_frames * n_mels floats; utterance u starts at frame_off[u] * n_mels in the chosen layout. */
int sept_logmel_f32(const float* wav_dev, const int64_t* utt_off_dev, const int64_t* frame_off_dev,
                    const int32_t* item_off_dev, int n_utts, int n_fft, int hop, int n_mels, int deriv, int layout,
                    float* out_dev, sept_stream_t stream);

/* Waveform gradient of the frame-major, deriv-0 log-mel of sept_logmel_f32 (the gradient torchaudio's MelSpectrogram +
 * AmplitudeToDB give under autograd): dwav = d(sum_{f,b} grad[f,b] * logmel[f,b]) / d wav, where grad_dev holds
 * total_frames * n_mels floats in the frame-major layout.  The clamp at 1e-10 passes no gradient (bands of zero power
 * give exactly 0).  Writes dwav for every sample of every utterance (samples outside all utterances are untouched).
 * n_items = item_off[n_utts]; workspace_dev holds sept_logmel_bwd_workspace_bytes(n_fft, hop, n_items) bytes (16-byte
 * aligned; about 0.46 GB per audio-hour at n_fft 800, hop 160).  Accepts every (n_fft, hop, n_mels) sept_logmel_f32
 * accepts.  Deterministic (no atomics), no allocation, capturable. */
size_t sept_logmel_bwd_workspace_bytes(int n_fft, int hop, int64_t n_items);
int sept_logmel_bwd_f32(const float* wav_dev, const int64_t* utt_off_dev, const int64_t* frame_off_dev,
                        const int32_t* item_off_dev, int n_utts, int64_t n_items, int n_fft, int hop, int n_mels,
                        const float* grad_dev, void* workspace_dev, float* dwav_dev, sept_stream_t stream);

/* MFCC-40 of the waveform, of np.gradient(waveform) and of np.gradient(waveform, 2).  Replaces mfcc(audio)
 * (feature_extraction/audio_feature_extraction.py:15-26 -> torchaudio/transforms/_transforms.py:634-718): n_fft 400,
 * hop 200, 128 mels, dB with top_db = 80 below the per-utterance maximum, orthonormal DCT-II.
 * Layouts must come from sept_extract_layout(n_fft=400, hop=200).
 * scratch_dev: total_frames * 257 floats (two mel-power streams + a frame->utterance map); utt_max_dev: 2 * n_utts
 * int32 (the call zeroes it);
 * out_dev: total_frames * 120 floats, utterance u is a (120, T_u) block at frame_off[u] * 120. */
int sept_mfcc_f32(const float* wav_dev, const int64_t* utt_off_dev, const int64_t* frame_off_dev,
                  const int32_t* item_off_dev, int n_utts, int64_t total_frames, float* scratch_dev,
                  int32_t* utt_max_dev, float* out_dev, sept_stream_t stream);

/* Waveform gradient of sept_mfcc_f32 (what torch autograd gives through torchaudio's MFCC for the three streams of
 * mfcc(audio): x, np.gradient(x), np.gradient(x, 2)): dwav = d(sum grad * mfcc) / d wav, where grad_dev holds
 * total_frames * 120 floats in sept_mfcc_f32's (120, T_u) block layout.  The top_db floor sends the gradient of every
 * floored value to the utterance's maximum (split evenly among tied maxima), the clamp at 1e-10 passes none.  Layouts
 * from sept_extract_layout(n_fft = 400, hop = 200); n_items = item_off[n_utts].  Writes dwav for every sample of every
 * utterance (samples outside all utterances are untouched).  workspace_dev holds
 * sept_mfcc_bwd_workspace_bytes(n_utts, total_frames, n_items) bytes, 16-byte aligned: 2876 bytes per frame plus 8 per
 * utterance, about 0.83 GB per audio-hour (288 000 frames), computed from the shapes.  Recomputes the mel power from
 * the waveform; deterministic (no atomics), no allocation, capturable. */
size_t sept_mfcc_bwd_workspace_bytes(int n_utts, int64_t total_frames, int64_t n_items);
int sept_mfcc_bwd_f32(const float* wav_dev, const int64_t* utt_off_dev, const int64_t* frame_off_dev,
                      const int32_t* item_off_dev, int n_utts, int64_t total_frames, int64_t n_items,
                      const float* grad_dev, void* workspace_dev, float* dwav_dev, sept_stream_t stream);

/* ---- resampling ahead of extraction --------------------------------------------------------------------------------
 * Band-limited sinc resampling of a ragged batch.  Replaces torchaudio.transforms.Resample(sample_rate, 16000) as the
 * reference applies it to the 44.1 kHz MSP-Improv corpus (feature_extraction/audio_feature_extraction.py:139-141 ->
 * torchaudio/functional/functional.py _get_sinc_resample_kernel/_apply_sinc_resample_kernel: sinc_interp_hann,
 * lowpass_filter_width 6, rolloff 0.99).  Rates are reduced by their gcd to orig/up; at most 4096 of each
 * (SEPT_E_UNSUPPORTED beyond).  Output length per utterance of n samples is torchaudio's:
 * min(ceil(float32(up * n / orig)), (n / orig + 1) * up), the quotient taken in double, as Python's int / int, and
 * rounded to float32, the default dtype torch.as_tensor gives it, before the ceil.  So it can differ by one either way
 * from the exact ceil(up * n / orig); the second term is the number of samples torchaudio's conv1d produces. */

/* HOST helper: out_off_host[n_utts+1] from in_off_host[n_utts+1].  SEPT_E_BADARG for decreasing offsets and for an
 * utterance with up * n >= 2^53, where the double quotient would no longer be Python's. */
int sept_resample_layout(const int64_t* in_off_host, int n_utts, int orig_freq, int new_freq, int64_t* out_off_host);

int sept_resample_f32(const float* in_dev, const int64_t* in_off_dev, const int64_t* out_off_dev, int n_utts,
                      int64_t total_out, int orig_freq, int new_freq, float* out_dev, sept_stream_t stream);

/* 16-bit PCM -> float32 in [-1, 1): out = pcm / 32768, the normalisation torchaudio.load applies before the reference's
 * callables see the audio (feature_extraction/audio_feature_extraction.py:182); lets bulk jobs copy half the bytes. */
int sept_pcm16_to_f32(const int16_t* pcm_dev, int64_t n, float* out_dev, sept_stream_t stream);

/* ---- per-speaker normalisation (preprocess_data/preprocess_adversary_data.py:26-27, 41-48, 357-385) -------------
 * feat_dev: (total_frames, n_feat) frame-major features; a frame that lies in k training windows (win_len, shift_len)
 * counts k times, utterances flagged in whole_dev (test split) count every frame once.
 * spk_ptr/spk_utts: CSR list of utterance ids per speaker.  utt_partial_dev: workspace n_utts*5*n_feat floats.
 * stats_dev: (n_spk, 5, n_feat) = count, mean, std (ddof 0), min, max. */
int sept_speaker_stats_f32(const float* feat_dev, const int64_t* frame_off_dev, const uint8_t* whole_dev, int n_utts,
                           int n_feat, int win_len, int shift_len, const int32_t* spk_ptr_dev,
                           const int32_t* spk_utts_dev, int n_spk, float* utt_partial_dev, float* stats_dev,
                           sept_stream_t stream);

/* znorm (x-mean)/(std+1e-5) or min_max (x-min)/(max-min)*2-1 of every frame with its speaker's statistics (:377-381);
 * out_dev (total_frames, n_feat). */
int sept_normalize_f32(const float* feat_dev, const int64_t* frame_off_dev, const int32_t* spk_of_utt_dev,
                       const float* stats_dev, int n_utts, int n_feat, int mode, float* out_dev, sept_stream_t stream);

/* Same, gathered into training windows: window w covers frames win_t0[w] .. +win_len of utterance win_utt[w]; rows past
 * the utterance end are the normalised zero padding of :29-35.  out_dev (n_windows, win_len, n_feat) -- the
 * (B, 1, 200, 128) batches the cloak layer consumes. */
int sept_normalize_windows_f32(const float* feat_dev, const int64_t* frame_off_dev, const int32_t* spk_of_utt_dev,
                               const float* stats_dev, const int32_t* win_utt_dev, const int32_t* win_t0_dev,
                               int n_windows, int win_len, int n_feat, int mode, float* out_dev, sept_stream_t stream);

/* Backward of sept_normalize_windows_f32 (utt_win_ptr_dev != NULL) or of sept_normalize_f32 (utt_win_ptr_dev == NULL):
 * what torch autograd gives for sum(grad * out) through the reference's normalisation, padded rows included.
 * grad_dev is laid out like the forward's out_dev.  Window mode: window w covers frames win_t0[w] .. +win_len of the
 * utterance whose CSR list holds it: utt_win_dev[utt_win_ptr[u] .. utt_win_ptr[u+1]) are the windows of utterance u
 * sorted by (win_t0, window index) (any table works: subsets, any order, repeated windows; win_t0 >= 0).
 * dfeat_dev (total_frames, n_feat) or NULL: every frame is written (0 for frames in no window).
 * dstats_dev (n_spk, 5, n_feat) or NULL: the gradient of the statistics (count row 0; znorm fills mean and std, min_max
 * min and max); needs spk_ptr/spk_utts (the CSR of sept_speaker_stats_f32) and workspace_dev of
 * sept_normalize_bwd_workspace_bytes(n_utts, n_feat) bytes.  Deterministic (no atomics), no allocation, capturable. */
size_t sept_normalize_bwd_workspace_bytes(int n_utts, int n_feat);
int sept_normalize_bwd_f32(const float* feat_dev, const int64_t* frame_off_dev, const int32_t* spk_of_utt_dev,
                           const float* stats_dev, const int32_t* win_t0_dev, const int32_t* utt_win_ptr_dev,
                           const int32_t* utt_win_dev, int n_windows, int win_len, int n_utts, int n_feat, int mode,
                           const float* grad_dev, const int32_t* spk_ptr_dev, const int32_t* spk_utts_dev, int n_spk,
                           void* workspace_dev, float* dfeat_dev, float* dstats_dev, sept_stream_t stream);

/* Backward of sept_speaker_stats_f32 (what torch autograd gives through the reference's stacked-rows mean, ddof-0 std,
 * min and max), in two calls, on one rank or on several (each rank holding some of a speaker's utterances).  Every rank
 * passes the same stats_dev (the forward's result; merged over the ranks when there are several) with the same n_spk
 * speaker rows, the CSR of its own utterances over those rows (a speaker the rank does not hold is an empty range and gets
 * tie weight 0) and spk_of_utt_dev [n_utts], the speaker row of each of its utterances.
 * _ties_i32 writes ties_dev (n_spk, 2, n_feat) int32: the summed window multiplicity of the rank's frames equal to each
 * speaker's min (row 0) and max (row 1).  workspace_dev holds sept_speaker_stats_bwd_ties_workspace_bytes(n_utts, n_feat)
 * bytes, 16-byte aligned.  With several ranks, sum ties_dev over the ranks (exact in int32) and dstats_dev over the ranks
 * before the second call.
 * _frames_f32 writes dfeat_dev (total_frames, n_feat) = d(sum dstats * stats) / d feat for every frame (0 for frames in
 * no training window).  Row 0 (count) of dstats_dev is ignored.  The min / max gradient goes to the frames equal to it in
 * proportion to their window multiplicity (ties_dev).  Where the forward's std is exactly 0 (every weighted value of that
 * speaker and feature equal, e.g. digital silence) no gradient flows through the std (sqrt's derivative there is 0 * inf
 * in torch).  Deterministic, no allocation, capturable. */
size_t sept_speaker_stats_bwd_ties_workspace_bytes(int n_utts, int n_feat);
int sept_speaker_stats_bwd_ties_i32(const float* feat_dev, const int64_t* frame_off_dev, const uint8_t* whole_dev,
                                    int n_utts, int n_feat, int win_len, int shift_len, const int32_t* spk_of_utt_dev,
                                    const int32_t* spk_ptr_dev, const int32_t* spk_utts_dev, int n_spk,
                                    const float* stats_dev, void* workspace_dev, int32_t* ties_dev, sept_stream_t stream);
int sept_speaker_stats_bwd_frames_f32(const float* feat_dev, const int64_t* frame_off_dev, const uint8_t* whole_dev,
                                      int n_utts, int n_feat, int win_len, int shift_len, const int32_t* spk_of_utt_dev,
                                      const float* stats_dev, const float* dstats_dev, const int32_t* ties_dev,
                                      float* dfeat_dev, sept_stream_t stream);

/* ---- cloak noise layer + gradient reversal -------------------------------------------------------------------------
 * Forward of cloak_noise (model/cloak_models.py:41-58): out = x*mask + locs + sigma(rhos) * eps*mask with
 * sigma = (1 + tanh rho)/2 * (max_scale - min_scale) + min_scale, broadcast over the batch.  eps_dev != NULL supplies
 * the noise sample; otherwise it is drawn on the device as eps_std * N(0,1) from Philox4x32-10(seed, offset) (the
 * reference draws Normal(0, 0.1) on the CPU, :37,47).  draw_dev (may be NULL) is a device counter of draws so far: the
 * Philox offset becomes offset + *draw_dev * ceil(wf/4), which lets a CUDA graph that contains this call produce a fresh
 * sample on every replay (advance it with sept_counter_add_u64 inside the same graph).  per_sample = 1 gives every batch
 * element its own eps (eps_dev / eps_out_dev are then (batch, wf), draw index *draw_dev + b): the batched equivalent of
 * the reference's evaluation loop that calls the layer once per window (training/adversary_cloak_evaluation.py:73-83);
 * forward only.  mask_dev, eps_out_dev, noise_out_dev may be NULL.  wf = W*F must be a multiple of 4. */
int sept_cloak_fwd_f32(const float* x_dev, const float* locs_dev, const float* rhos_dev, const float* mask_dev,
                       const float* eps_dev, uint64_t seed, uint64_t offset, const uint64_t* draw_dev, int per_sample,
                       float eps_std, float min_scale, float max_scale, int batch, int wf, float* out_dev,
                       float* eps_out_dev, float* noise_out_dev, sept_stream_t stream);

/* *counter_dev += inc on the stream (one thread); keeps the draw counter of sept_cloak_fwd_f32 on the device. */
int sept_counter_add_u64(uint64_t* counter_dev, uint64_t inc, sept_stream_t stream);

/* workspace of the backward, in bytes, for a (batch, wf) problem; zero it once, the kernel leaves it reusable */
size_t sept_cloak_bwd_workspace_bytes(int wf);

/* Backward of the cloak layer fused with gradient reversal (model/reversal_gradient.py:19-23):
 * g = g_a - lambda * g_b (g_b may be NULL); dlocs = sum_b g; drhos = sum_b g * eps*mask * dsigma/drho; dx = g*mask.
 * drhos_dev and dx_dev may be NULL.  Deterministic. */
int sept_cloak_grl_bwd_f32(const float* g_a_dev, const float* g_b_dev, float lambda, const float* eps_dev,
                           const float* rhos_dev, const float* mask_dev, float min_scale, float max_scale, int batch,
                           int wf, void* workspace_dev, float* dlocs_dev, float* drhos_dev, float* dx_dev,
                           sept_stream_t stream);

/* Backward of GradientReversalFunction (model/reversal_gradient.py:19-23): dx = -lambda * g. */
int sept_grl_bwd_f32(const float* g_dev, float lambda, int64_t n, float* dx_dev, sept_stream_t stream);

/* ---- waveform-domain cloak ----------------------------------------------------------------------------------------
 * The signal-domain counterpart of cloak_noise: a learned noise of `period` samples (noise = locs + sigma(rhos) * eps,
 * drawn by sept_cloak_fwd_f32 with batch = 0, wf = period) is tiled over every utterance of a ragged batch from the
 * utterance's first sample: y[s] = x[s] + noise[(s - utt_off[u]) mod period].  Tile k of utterance u is its period
 * utt_off[u] + k*period .. + period, clipped to the utterance.  period must be a multiple of 4; every utterance must be
 * shorter than 2^31 samples and 0 <= utt_off[0] <= ... <= utt_off[n_utts] <= n_samples (sept_wave_cloak_layout checks
 * both on the host). */

/* HOST helper: tile_off_host[n_utts+1], the tiles of utterance u being tile_off[u] .. tile_off[u+1]-1
 * (ceil(length / period) each); validates the offsets as above. */
int sept_wave_cloak_layout(const int64_t* utt_off_host, int n_utts, int period, int64_t* tile_off_host);

/* y = x + noise tiled over every utterance; samples before utt_off[0] and from utt_off[n_utts] to n_samples are copied.
 * x_dev, y_dev (n_samples) and noise_dev (period) 16-byte aligned. */
int sept_wave_cloak_fwd_f32(const float* x_dev, const int64_t* utt_off_dev, int n_utts, int64_t n_samples,
                            const float* noise_dev, int period, float* y_dev, sept_stream_t stream);

/* Evaluation with fresh noise per utterance: y[s] = x[s] + (locs[j] + sigma(rhos[j]) * eps_u[j]) for every sample s of
 * utterance u, j = (s - utt_off[u]) mod period; samples before utt_off[0] and from utt_off[n_utts] to n_samples are
 * copied.  The sum and the product are rounded separately, as in sept_cloak_fwd_f32.  eps_u is generated inside the kernel;
 * no (n_utts, period) buffer is written.
 * Draw rule (L = period): utterance u uses draw index d_u = (*draw_dev or 0) + utt_draw[u], or + u when utt_draw_dev
 * is NULL. eps_u is bit for bit row d_u of what sept_cloak_fwd_f32(per_sample = 1, wf = L) draws: component j % 4 of
 * normal4(seed, offset + d_u * ceil(L/4), j / 4, eps_std). It is the same Philox stream and the same (seed, offset, draw)
 * rules as every other draw in the library.
 * With global utterance ids in utt_draw_dev (int64, n_utts; the caller keeps them distinct and non-negative), an
 * utterance's noisy audio depends neither on its batch, nor on its position in the batch, nor on the rank that holds it.
 * The call does not advance *draw_dev (sept_counter_add_u64 does).  eps_dev (n_utts, period), indexed by batch position
 * u, replaces the draw; it may be NULL.  workspace_dev holds sept_wave_cloak_eval_workspace_bytes(period) bytes (sigma of
 * every phase, written by the call).  x_dev, y_dev, locs_dev, rhos_dev, eps_dev and workspace_dev 16-byte aligned; period
 * and the offsets as above.  No atomics, no allocation, capturable. */
size_t sept_wave_cloak_eval_workspace_bytes(int period);
int sept_wave_cloak_eval_f32(const float* x_dev, const int64_t* utt_off_dev, int n_utts, int64_t n_samples,
                             const float* locs_dev, const float* rhos_dev, const float* eps_dev,
                             uint64_t seed, uint64_t offset, const uint64_t* draw_dev, const int64_t* utt_draw_dev,
                             float eps_std, float min_scale, float max_scale, int period,
                             void* workspace_dev, float* y_dev, sept_stream_t stream);

/* Backward of sept_wave_cloak_fwd_f32 with respect to the noise: r[j] = the sum of g over every in-utterance sample of
 * phase j, r_dev (period).  dx = g needs no call; dlocs = r and drhos = r * eps * dsigma/drho follow from
 * sept_cloak_grl_bwd_f32(g_a = r, batch = 1, mask = NULL).  tile_off_dev is sept_wave_cloak_layout's table on the device,
 * n_tiles = tile_off[n_utts].  workspace_dev holds sept_wave_cloak_bwd_workspace_bytes(period) bytes (592 partial rows
 * of the period, 16-byte aligned); g_dev and r_dev 16-byte aligned.  Deterministic: no atomics, a fixed summation order
 * that does not depend on the GPU (DESIGN 3.3b); no allocation, capturable. */
size_t sept_wave_cloak_bwd_workspace_bytes(int period);
int sept_wave_cloak_bwd_f32(const float* g_dev, const int64_t* utt_off_dev, const int64_t* tile_off_dev, int n_utts,
                            int64_t n_tiles, int period, void* workspace_dev, float* r_dev, sept_stream_t stream);

/* Backward of sept_wave_cloak_eval_f32 with respect to locs and rhos, for training with fresh noise per utterance:
 * dlocs[j] = the sum of g over every in-utterance sample of phase j (the bits of sept_wave_cloak_bwd_f32's r), and
 * drhos[j] = q[j] * dsigma/drho(rhos[j]), q[j] = the sum of g * eps_u[j] over the same samples, each product rounded on
 * its own and summed in the order of r (DESIGN 3.3d); dsigma/drho = (1 - tanh^2 rho) / 2 * (max_scale - min_scale), as
 * in sept_cloak_grl_bwd_f32.  dx = g needs no call.  eps_u follows sept_wave_cloak_eval_f32's draw rule with the same
 * (eps_dev, seed, offset, draw_dev, utt_draw_dev, eps_std) and is generated again inside the kernel, not stored.  The call
 * must receive the draw base its forward read: that forward's *draw_dev before sept_counter_add_u64 moved it (copy it
 * to a buffer of its own before the counter moves).  tile_off_dev and n_tiles as for sept_wave_cloak_bwd_f32.
 * workspace_dev holds sept_wave_cloak_bwd_per_utt_workspace_bytes(period) bytes (2 x 592 partial rows of the period);
 * g_dev, rhos_dev, eps_dev, workspace_dev, dlocs_dev and drhos_dev 16-byte aligned.  Deterministic: no atomics, and the
 * bits depend only on the layout and the draw inputs, not on the GPU; no allocation, capturable. */
size_t sept_wave_cloak_bwd_per_utt_workspace_bytes(int period);
int sept_wave_cloak_bwd_per_utt_f32(const float* g_dev, const int64_t* utt_off_dev, const int64_t* tile_off_dev,
                                    int n_utts, int64_t n_tiles, int period, const float* rhos_dev,
                                    const float* eps_dev, uint64_t seed, uint64_t offset, const uint64_t* draw_dev,
                                    const int64_t* utt_draw_dev, float eps_std, float min_scale, float max_scale,
                                    void* workspace_dev, float* dlocs_dev, float* drhos_dev, sept_stream_t stream);

/* Class-balance noise augmentation (preprocess_data/preprocess_adversary_data.py:392-421): job j adds to row
 * job_row[j] of data_dev (n_rows, row_elems) the noise samples draw_id[job_ptr[j] .. job_ptr[j+1]) in that order -- the
 * reference writes the noisy copy through an alias of the source window, so a window drawn m times carries the sum of its
 * m samples, shared by all its copies.  noise_dev NULL: sample t is N(0, std) from Philox(seed, t); else row t of
 * noise_dev (n_draws, row_elems).  Rows of different jobs must be distinct.  At most 65535 jobs per call. */
int sept_add_noise_rows_f32(float* data_dev, const int64_t* job_row_dev, const int32_t* job_ptr_dev,
                            const int64_t* draw_id_dev, int n_jobs, int row_elems, uint64_t seed, float std,
                            const float* noise_dev, sept_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SEPT_H_ */
