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
 * lowpass_filter_width 6, rolloff 0.99).  Output length per utterance: ceil(new_freq * n / orig_freq). */

/* HOST helper: out_off_host[n_utts+1] from in_off_host[n_utts+1]. */
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
