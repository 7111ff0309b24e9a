// C ABI of libsept_b200 (include/sept.h): argument checking, the per-device constant cache, kernel launches.
#include <cuda_runtime.h>
#include <cstdlib>

#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/sept.h"
#include "augment.h"
#include "cloak.h"
#include "extract.h"
#include "extract_bwd.h"
#include "extract_core.cuh"
#include "mfcc_bwd.h"
#include "norm.h"
#include "norm_bwd.h"
#include "resample.h"
#include "tables.h"
#include "wave_cloak.h"

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

int cuda_fail(cudaError_t e, const char* what) {
    return fail(SEPT_E_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

#define SEPT_CUDA(call)                                                  \
    do {                                                                 \
        cudaError_t e_ = (call);                                         \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);              \
    } while (0)

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- immutable per-(device, n_fft, n_mels) constants -------------------------------------------------------------
struct ExtractConsts {
    float* window = nullptr;
    float* tws = nullptr;
    sept::MelStep* mel_prog = nullptr;
    int n_mel_entries = 0, n_mel_head = 0, mel_fast = 0;
};

struct ResampleConsts {
    int32_t* k_lo = nullptr;
    float* w = nullptr;
    int taps = 0, width = 0;
    int32_t* tile_base = nullptr;
    float* tile_wt = nullptr;
    int n_groups = 0, tg = 0, base_min = 0, base_max = 0;
};

std::map<std::tuple<int, int, int>, ResampleConsts> g_resample;

std::mutex g_mu;
std::map<std::tuple<int, int, int>, ExtractConsts> g_consts;
std::map<int, float*> g_dct;
std::map<int, int> g_sm_count;

template <class T>
cudaError_t upload(const std::vector<T>& h, T** d) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(d), h.size() * sizeof(T) + 16);
    if (e != cudaSuccess) return e;
    return cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice);
}

int get_consts(int n_fft, int n_mels, ExtractConsts* out, int* sm_count) {
    int dev = 0;
    SEPT_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_sm_count.count(dev)) {
        int n = 0;
        SEPT_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
        g_sm_count[dev] = n;
    }
    *sm_count = g_sm_count[dev];
    auto key = std::make_tuple(dev, n_fft, n_mels);
    auto it = g_consts.find(key);
    if (it == g_consts.end()) {
        ExtractConsts c;
        std::vector<float> win = sept::make_hann_periodic(n_fft);
        std::vector<float> tws = sept::make_split_twiddles(n_fft);
        sept::MelProgram prog;
        sept::make_mel_program(n_fft, n_mels, 16000, prog);
        c.n_mel_entries = (int)prog.entries.size();
        c.n_mel_head = prog.n_head;
        c.mel_fast = sept::extract_mel_fast_ok(n_fft, n_mels, prog.n_head, prog.round_steps.data(), (int)prog.round_steps.size()) ? 1 : 0;
        SEPT_CUDA(upload(win, &c.window));
        SEPT_CUDA(upload(tws, &c.tws));
        SEPT_CUDA(upload(prog.entries, &c.mel_prog));
        it = g_consts.emplace(key, c).first;
    }
    *out = it->second;
    return SEPT_OK;
}

int get_dct(float** out) {
    int dev = 0;
    SEPT_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    auto it = g_dct.find(dev);
    if (it == g_dct.end()) {
        std::vector<float> d = sept::make_dct_ortho(40, 128);
        float* dd = nullptr;
        SEPT_CUDA(upload(d, &dd));
        it = g_dct.emplace(dev, dd).first;
    }
    *out = it->second;
    return SEPT_OK;
}

long long gcd_ll(long long a, long long b) { while (b) { const long long t = a % b; a = b; b = t; } return a; }

int get_resample(int orig, int up, ResampleConsts* out) {
    int dev = 0;
    SEPT_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_mu);
    auto key = std::make_tuple(dev, orig, up);
    auto it = g_resample.find(key);
    if (it == g_resample.end()) {
        ResampleConsts c;
        std::vector<int32_t> k_lo;
        std::vector<float> rows;
        c.width = sept::make_resample_rows(orig, up, k_lo, rows, c.taps);
        SEPT_CUDA(upload(k_lo, &c.k_lo));
        SEPT_CUDA(upload(rows, &c.w));
        sept::ResampleTiles tiles;
        sept::make_resample_tiles(up, c.taps, k_lo, rows, tiles);
        SEPT_CUDA(upload(tiles.base, &c.tile_base));
        SEPT_CUDA(upload(tiles.wt, &c.tile_wt));
        c.n_groups = tiles.n_groups; c.tg = tiles.tg; c.base_min = tiles.base_min; c.base_max = tiles.base_max;
        it = g_resample.emplace(key, c).first;
    }
    *out = it->second;
    return SEPT_OK;
}

bool supported_n_fft(int n_fft) { return n_fft == 400 || n_fft == 800 || n_fft == 1600; }

int check_extract_shape(int n_fft, int hop, int n_mels, int n_mel_entries) {
    if (!supported_n_fft(n_fft))
        return fail(SEPT_E_UNSUPPORTED, "n_fft=%d unsupported: the kernels cover 400, 800 and 1600 (2^a * 25)", n_fft);
    if (hop <= 0 || (hop & 1) || hop > n_fft)
        return fail(SEPT_E_UNSUPPORTED, "hop=%d unsupported: must be even and in (0, n_fft]", hop);
    if (n_mels <= 0 || n_mels > 512) return fail(SEPT_E_UNSUPPORTED, "n_mels=%d unsupported (1..512)", n_mels);
    if (n_mel_entries >= 0 && sept::extract_smem_bytes_for(n_fft, hop, n_mel_entries) > sept::kMaxDynSmem)
        return fail(SEPT_E_UNSUPPORTED, "n_fft=%d hop=%d n_mels=%d does not fit the 227 KB of shared memory", n_fft, hop,
                    n_mels);
    return SEPT_OK;
}

// the set-up of every extraction entry, forward or backward: the shape checks and the (n_fft, n_mels) constants
int extract_setup(int n_fft, int hop, int n_mels, ExtractConsts* c, int* sms) {
    int rc = check_extract_shape(n_fft, hop, n_mels, -1);
    if (rc) return rc;
    rc = get_consts(n_fft, n_mels, c, sms);
    if (rc) return rc;
    return check_extract_shape(n_fft, hop, n_mels, c->n_mel_entries);
}

// launch parameters shared by every extraction launch: the batch, its layout and the (n_fft, n_mels) constants.  A
// backward recomputes the forward with the same struct.
sept::ExtractParams extract_params(const ExtractConsts& c, const float* wav, const int64_t* utt_off,
                                   const int64_t* frame_off, const int32_t* item_off, int n_utts, int hop, int n_mels) {
    sept::ExtractParams p{};
    p.wav = wav; p.utt_off = utt_off; p.frame_off = frame_off; p.item_off = item_off;
    p.n_utts = n_utts; p.hop = hop; p.n_mels = n_mels; p.n_mel_entries = c.n_mel_entries; p.n_mel_head = c.n_mel_head; p.mel_fast = c.mel_fast;
    p.window = c.window; p.tws = c.tws; p.mel_prog = c.mel_prog;
    return p;
}

// The MFCC forward's power launch (p: extract_params at n_fft 400, hop 200, 128 mels): mel power of x and
// np.gradient(x) to p.out [2][total_frames][128], the bits of each utterance's largest value to p.utt_max [2][n_utts],
// the utterance of every frame to p.frame_utt.  It is deterministic, so the backward, which runs this same launch,
// recomputes the forward's values bit for bit.
int launch_mfcc_power(const sept::ExtractParams& p, int sms, cudaStream_t st) {
    SEPT_CUDA(cudaMemsetAsync(p.utt_max, 0, sizeof(int32_t) * 2 * (size_t)p.n_utts, st));
    SEPT_CUDA(sept::launch_extract(p, 400, sept::kModeMfccPower, sms, st));
    return SEPT_OK;
}

}  // namespace

extern "C" {

int sept_version(void) { return 200; }

#ifndef SEPT_SRC_HASH
#define SEPT_SRC_HASH "unknown"
#endif
/* the marker lets the loader read the hash out of the file without dlopen-ing a stale library */
const char* sept_source_hash(void) { return "SEPT_SRC_HASH=" SEPT_SRC_HASH; }

const char* sept_last_error(void) { return g_err.c_str(); }

int sept_init(int n_mels) {
    for (int n_fft : {400, 800, 1600}) {
        ExtractConsts c;
        int sms;
        int rc = get_consts(n_fft, n_mels, &c, &sms);
        if (rc) return rc;
    }
    float* d;
    return get_dct(&d);
}

int sept_frames_per_item(int n_fft) { return sept::extract_frames_per_item(n_fft); }

int sept_extract_layout(const int64_t* utt_off, int n_utts, int n_fft, int hop, int64_t* frame_off, int32_t* item_off) {
    if (!utt_off || !frame_off || !item_off || n_utts < 0) return fail(SEPT_E_BADARG, "sept_extract_layout: bad argument");
    int rc = check_extract_shape(n_fft, hop, 1, -1);
    if (rc) return rc;
    const int fpw = sept::extract_frames_per_item(n_fft);
    frame_off[0] = 0;
    item_off[0] = 0;
    for (int u = 0; u < n_utts; ++u) {
        const int64_t n = utt_off[u + 1] - utt_off[u];
        if (n <= n_fft / 2)
            return fail(SEPT_E_TOO_SHORT, "utterance %d has %lld samples; reflect padding of %d needs more", u, (long long)n,
                        n_fft / 2);
        if (n >= (int64_t)1 << 31) return fail(SEPT_E_BADARG, "utterance %d is longer than 2^31 samples", u);
        const int64_t T = 1 + n / hop;
        frame_off[u + 1] = frame_off[u] + T;
        const int64_t items = item_off[u] + (T + fpw - 1) / fpw;
        if (items >= (int64_t)1 << 31) return fail(SEPT_E_BADARG, "batch exceeds 2^31 work items; split it");
        item_off[u + 1] = (int32_t)items;
    }
    return SEPT_OK;
}

int sept_logmel_f32(const float* wav, const int64_t* utt_off, const int64_t* frame_off, const int32_t* item_off,
                    int n_utts, int n_fft, int hop, int n_mels, int deriv, int layout, float* out, sept_stream_t stream) {
    if (n_utts == 0) return SEPT_OK;
    if (!wav || !utt_off || !frame_off || !item_off || !out || n_utts < 0)
        return fail(SEPT_E_BADARG, "sept_logmel_f32: null pointer or negative n_utts");
    if (layout != SEPT_LAYOUT_FRAME_MAJOR && layout != SEPT_LAYOUT_BAND_MAJOR)
        return fail(SEPT_E_BADARG, "sept_logmel_f32: layout %d", layout);
    ExtractConsts c;
    int sms = 0;
    int rc = extract_setup(n_fft, hop, n_mels, &c, &sms);
    if (rc) return rc;
    sept::ExtractParams p = extract_params(c, wav, utt_off, frame_off, item_off, n_utts, hop, n_mels);
    p.deriv = deriv ? 1 : 0;
    p.out = out;
    const int mode = layout == SEPT_LAYOUT_FRAME_MAJOR ? sept::kModeDbFrameMajor : sept::kModeDbBandMajor;
    SEPT_CUDA(sept::launch_extract(p, n_fft, mode, sms, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_logmel_bwd_workspace_bytes(int n_fft, int hop, int64_t n_items) {
    return sept::logmel_bwd_workspace_bytes(n_fft, hop, n_items);
}

int sept_logmel_bwd_f32(const float* wav, const int64_t* utt_off, const int64_t* frame_off, const int32_t* item_off,
                        int n_utts, int64_t n_items, int n_fft, int hop, int n_mels, const float* grad, void* workspace,
                        float* dwav, sept_stream_t stream) {
    if (n_utts == 0 || n_items == 0) return SEPT_OK;
    if (!wav || !utt_off || !frame_off || !item_off || !grad || !workspace || !dwav || n_utts < 0 || n_items < 0)
        return fail(SEPT_E_BADARG, "sept_logmel_bwd_f32: null pointer or negative size");
    if (!aligned16(workspace)) return fail(SEPT_E_BADARG, "sept_logmel_bwd_f32: workspace must be 16-byte aligned");
    ExtractConsts c;
    int sms = 0;
    int rc = extract_setup(n_fft, hop, n_mels, &c, &sms);
    if (rc) return rc;
    sept::LogmelBwdParams p{};
    p.f = extract_params(c, wav, utt_off, frame_off, item_off, n_utts, hop, n_mels);
    p.n_items = n_items; p.grad = grad; p.ws = static_cast<float*>(workspace); p.dwav = dwav;
    SEPT_CUDA(sept::launch_logmel_bwd(p, n_fft, sms, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_mfcc_f32(const float* wav, const int64_t* utt_off, const int64_t* frame_off, const int32_t* item_off, int n_utts,
                  int64_t total_frames, float* scratch, int32_t* utt_max, float* out, sept_stream_t stream) {
    if (n_utts == 0) return SEPT_OK;
    if (!wav || !utt_off || !frame_off || !item_off || !scratch || !utt_max || !out || n_utts < 0 || total_frames <= 0)
        return fail(SEPT_E_BADARG, "sept_mfcc_f32: null pointer or bad size");
    ExtractConsts c;
    int sms = 0;
    int rc = extract_setup(400, 200, 128, &c, &sms);
    if (rc) return rc;
    float* dct = nullptr;
    rc = get_dct(&dct);
    if (rc) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    sept::ExtractParams p = extract_params(c, wav, utt_off, frame_off, item_off, n_utts, 200, 128);
    p.total_frames = total_frames; p.out = scratch; p.utt_max = utt_max;
    p.frame_utt = reinterpret_cast<int*>(scratch + 2 * (size_t)total_frames * 128);
    rc = launch_mfcc_power(p, sms, st);
    if (rc) return rc;
    sept::MfccDctParams d{};
    d.power = scratch; d.utt_max = utt_max; d.frame_utt = p.frame_utt; d.frame_off = frame_off; d.dct = dct; d.n_utts = n_utts;
    d.total_frames = total_frames; d.top_db = 80.0f; d.out = out;
    SEPT_CUDA(sept::launch_mfcc_dct(d, st));
    return SEPT_OK;
}

size_t sept_mfcc_bwd_workspace_bytes(int n_utts, int64_t total_frames, int64_t n_items) {
    return sept::mfcc_bwd_layout(n_utts, total_frames, n_items).bytes;
}

int sept_mfcc_bwd_f32(const float* wav, const int64_t* utt_off, const int64_t* frame_off, const int32_t* item_off,
                      int n_utts, int64_t total_frames, int64_t n_items, const float* grad, void* workspace, float* dwav,
                      sept_stream_t stream) {
    if (n_utts == 0) return SEPT_OK;
    if (!wav || !utt_off || !frame_off || !item_off || !grad || !workspace || !dwav || n_utts < 0 || total_frames <= 0 ||
        n_items <= 0)
        return fail(SEPT_E_BADARG, "sept_mfcc_bwd_f32: null pointer or bad size");
    if (!aligned16(workspace)) return fail(SEPT_E_BADARG, "sept_mfcc_bwd_f32: workspace must be 16-byte aligned");
    ExtractConsts c;
    int sms = 0;
    int rc = extract_setup(400, 200, 128, &c, &sms);
    if (rc) return rc;
    float* dct = nullptr;
    rc = get_dct(&dct);
    if (rc) return rc;
    const sept::MfccBwdLayout l = sept::mfcc_bwd_layout(n_utts, total_frames, n_items);
    unsigned char* ws = static_cast<unsigned char*>(workspace);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    sept::MfccBwdParams b{};
    sept::ExtractParams& p = b.frames.f;                         // the power launch, then the frame passes' recompute
    p = extract_params(c, wav, utt_off, frame_off, item_off, n_utts, 200, 128);
    p.total_frames = total_frames; p.out = reinterpret_cast<float*>(ws + l.power);
    p.utt_max = reinterpret_cast<int32_t*>(ws + l.utt_max); p.frame_utt = reinterpret_cast<int*>(ws + l.frame_utt);
    rc = launch_mfcc_power(p, sms, st);
    if (rc) return rc;
    b.frames.n_items = n_items;
    b.grad = grad; b.dct = dct; b.frame_utt = p.frame_utt; b.utt_max = p.utt_max; b.total_frames = total_frames;
    b.power = p.out; b.part = reinterpret_cast<float*>(ws + l.part); b.amask = reinterpret_cast<uint32_t*>(ws + l.amask);
    b.rows0 = reinterpret_cast<float*>(ws + l.rows0); b.rows1 = reinterpret_cast<float*>(ws + l.rows1); b.dwav = dwav;
    SEPT_CUDA(sept::launch_mfcc_bwd(b, sms, st));
    return SEPT_OK;
}

int sept_resample_layout(const int64_t* in_off, int n_utts, int orig_freq, int new_freq, int64_t* out_off) {
    if (!in_off || !out_off || n_utts < 0 || orig_freq <= 0 || new_freq <= 0)
        return fail(SEPT_E_BADARG, "sept_resample_layout: bad argument");
    const long long g = gcd_ll(orig_freq, new_freq), orig = orig_freq / g, up = new_freq / g;
    if (orig > 4096 || up > 4096)
        return fail(SEPT_E_UNSUPPORTED, "sept_resample_layout: %d -> %d reduces to %lld/%lld, beyond the 4096-phase table limit",
                    orig_freq, new_freq, up, orig);
    out_off[0] = 0;
    for (int u = 0; u < n_utts; ++u) {
        const long long n = in_off[u + 1] - in_off[u];
        if (n < 0) return fail(SEPT_E_BADARG, "sept_resample_layout: offsets must be non-decreasing");
        // torchaudio's _apply_sinc_resample_kernel cuts at ceil(torch.as_tensor(new * length / orig)): Python's double
        // quotient, rounded to the default dtype float32 before the ceil, and at most the (n / orig + 1) * up samples its
        // conv1d produces.  The double quotient below is Python's while up * n < 2^53.
        if (n > ((1LL << 53) - 1) / up)
            return fail(SEPT_E_BADARG, "sept_resample_layout: utterance %d has %lld samples, too many for the length rule", u, n);
        const long long cut = (long long)ceilf((float)((double)(up * n) / (double)orig));
        const long long conv = (n / orig + 1) * up;
        const long long len = cut < conv ? cut : conv;
        if (out_off[u] > INT64_MAX - len) return fail(SEPT_E_BADARG, "sept_resample_layout: total output length overflows");
        out_off[u + 1] = out_off[u] + len;
    }
    return SEPT_OK;
}

int sept_resample_f32(const float* in, const int64_t* in_off, const int64_t* out_off, int n_utts, int64_t total_out,
                      int orig_freq, int new_freq, float* out, sept_stream_t stream) {
    if (n_utts == 0 || total_out == 0) return SEPT_OK;
    if (!in || !in_off || !out_off || !out || n_utts < 0 || total_out < 0 || orig_freq <= 0 || new_freq <= 0)
        return fail(SEPT_E_BADARG, "sept_resample_f32: bad argument");
    const long long g = gcd_ll(orig_freq, new_freq), orig = orig_freq / g, up = new_freq / g;
    if (orig > 4096 || up > 4096)
        return fail(SEPT_E_UNSUPPORTED, "sept_resample_f32: %d -> %d reduces to %lld/%lld, beyond the 4096-phase table limit",
                    orig_freq, new_freq, up, orig);
    ResampleConsts c;
    int rc = get_resample((int)orig, (int)up, &c);
    if (rc) return rc;
    sept::ResampleParams p{};
    p.in = in; p.in_off = in_off; p.out_off = out_off; p.n_utts = n_utts; p.orig = (int)orig; p.up = (int)up;
    p.width = c.width; p.taps = c.taps; p.k_lo = c.k_lo; p.w = c.w; p.out = out; p.total_out = total_out;
    static const bool simple_only = getenv("SEPT_RESAMPLE_SIMPLE") != nullptr;   // A/B and tests of the fallback kernel
    if (!simple_only) {
        p.tile_base = c.tile_base; p.tile_wt = c.tile_wt; p.n_groups = c.n_groups; p.tg = c.tg;
        p.base_min = c.base_min; p.base_max = c.base_max;
    }
    SEPT_CUDA(sept::launch_resample(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_pcm16_to_f32(const int16_t* pcm, int64_t n, float* out, sept_stream_t stream) {
    if (n == 0) return SEPT_OK;
    if (!pcm || !out || n < 0) return fail(SEPT_E_BADARG, "sept_pcm16_to_f32: bad argument");
    SEPT_CUDA(sept::launch_pcm16_to_f32(pcm, n, out, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_speaker_stats_f32(const float* feat, const int64_t* frame_off, const uint8_t* whole, int n_utts, int n_feat,
                           int win_len, int shift_len, const int32_t* spk_ptr, const int32_t* spk_utts, int n_spk,
                           float* utt_partial, float* stats, sept_stream_t stream) {
    if (!feat || !frame_off || !spk_ptr || !spk_utts || !utt_partial || !stats || n_utts < 0 || n_spk < 0 || n_feat <= 0 ||
        win_len <= 0 || shift_len <= 0)
        return fail(SEPT_E_BADARG, "sept_speaker_stats_f32: bad argument");
    sept::SpeakerStatsParams p{};
    p.feat = feat; p.frame_off = frame_off; p.whole = whole; p.n_utts = n_utts; p.n_feat = n_feat;
    p.win_len = win_len; p.shift_len = shift_len; p.utt_partial = utt_partial; p.spk_ptr = spk_ptr;
    p.spk_utts = spk_utts; p.n_spk = n_spk; p.stats = stats;
    SEPT_CUDA(sept::launch_speaker_stats(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_normalize_f32(const float* feat, const int64_t* frame_off, const int32_t* spk_of_utt, const float* stats,
                       int n_utts, int n_feat, int mode, float* out, sept_stream_t stream) {
    if (!feat || !frame_off || !spk_of_utt || !stats || !out || n_utts < 0 || n_feat <= 0 ||
        (mode != SEPT_NORM_ZNORM && mode != SEPT_NORM_MINMAX))
        return fail(SEPT_E_BADARG, "sept_normalize_f32: bad argument");
    sept::NormalizeParams p{};
    p.feat = feat; p.frame_off = frame_off; p.spk_of_utt = spk_of_utt; p.stats = stats; p.n_feat = n_feat;
    p.mode = mode; p.n_utts = n_utts; p.out = out;
    SEPT_CUDA(sept::launch_normalize(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_normalize_windows_f32(const float* feat, const int64_t* frame_off, const int32_t* spk_of_utt,
                               const float* stats, const int32_t* win_utt, const int32_t* win_t0, int n_windows,
                               int win_len, int n_feat, int mode, float* out, sept_stream_t stream) {
    if (!feat || !frame_off || !spk_of_utt || !stats || !win_utt || !win_t0 || !out || n_windows < 0 || win_len <= 0 ||
        n_feat <= 0 || (mode != SEPT_NORM_ZNORM && mode != SEPT_NORM_MINMAX))
        return fail(SEPT_E_BADARG, "sept_normalize_windows_f32: bad argument");
    sept::NormalizeParams p{};
    p.feat = feat; p.frame_off = frame_off; p.spk_of_utt = spk_of_utt; p.stats = stats; p.n_feat = n_feat;
    p.mode = mode; p.win_utt = win_utt; p.win_t0 = win_t0; p.n_windows = n_windows; p.win_len = win_len; p.out = out;
    SEPT_CUDA(sept::launch_normalize(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_normalize_bwd_workspace_bytes(int n_utts, int n_feat) {
    return n_utts > 0 && n_feat > 0 ? sept::normalize_bwd_workspace_bytes(n_utts, n_feat) : 0;
}

int sept_normalize_bwd_f32(const float* feat, const int64_t* frame_off, const int32_t* spk_of_utt, const float* stats,
                           const int32_t* win_t0, const int32_t* utt_win_ptr, const int32_t* utt_win, int n_windows,
                           int win_len, int n_utts, int n_feat, int mode, const float* grad, const int32_t* spk_ptr,
                           const int32_t* spk_utts, int n_spk, void* workspace, float* dfeat, float* dstats,
                           sept_stream_t stream) {
    const bool window = utt_win_ptr != nullptr;
    if (!feat || !frame_off || !spk_of_utt || !stats || !grad || (!dfeat && !dstats) || n_utts < 0 || n_feat <= 0 ||
        (window && (!win_t0 || !utt_win || n_windows < 0 || win_len <= 0)) ||
        (mode != SEPT_NORM_ZNORM && mode != SEPT_NORM_MINMAX))
        return fail(SEPT_E_BADARG, "sept_normalize_bwd_f32: bad argument");
    if (dstats && (!spk_ptr || !spk_utts || n_spk < 0 || !workspace))
        return fail(SEPT_E_BADARG, "sept_normalize_bwd_f32: dstats needs spk_ptr, spk_utts and the workspace");
    sept::NormalizeBwdParams p{};
    p.f.feat = feat; p.f.frame_off = frame_off; p.f.spk_of_utt = spk_of_utt; p.f.stats = stats; p.f.n_feat = n_feat;
    p.f.mode = mode; p.f.n_utts = n_utts;
    if (window) {
        p.f.win_utt = utt_win;                                   // non-null selects the window mode, as in the forward
        p.f.win_t0 = win_t0; p.f.n_windows = n_windows; p.f.win_len = win_len;
        p.utt_win_ptr = utt_win_ptr; p.utt_win = utt_win;
    }
    p.grad = grad; p.dfeat = dfeat;
    if (dstats) {
        p.upart = static_cast<float*>(workspace); p.spk_ptr = spk_ptr; p.spk_utts = spk_utts; p.n_spk = n_spk;
        p.dstats = dstats;
    }
    SEPT_CUDA(sept::launch_normalize_bwd(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_speaker_stats_bwd_ties_workspace_bytes(int n_utts, int n_feat) {
    return n_utts >= 0 && n_feat > 0 ? sept::speaker_stats_bwd_ties_workspace_bytes(n_utts, n_feat) : 0;
}

int sept_speaker_stats_bwd_ties_i32(const float* feat, const int64_t* frame_off, const uint8_t* whole, int n_utts,
                                    int n_feat, int win_len, int shift_len, const int32_t* spk_of_utt,
                                    const int32_t* spk_ptr, const int32_t* spk_utts, int n_spk, const float* stats,
                                    void* workspace, int32_t* ties, sept_stream_t stream) {
    if (!feat || !frame_off || !spk_of_utt || !spk_ptr || !spk_utts || !stats || !workspace || !ties || n_utts < 0 ||
        n_spk < 0 || n_feat <= 0 || win_len <= 0 || shift_len <= 0)
        return fail(SEPT_E_BADARG, "sept_speaker_stats_bwd_ties_i32: bad argument");
    if (!aligned16(workspace))
        return fail(SEPT_E_BADARG, "sept_speaker_stats_bwd_ties_i32: workspace must be 16-byte aligned");
    sept::SpeakerStatsBwdParams p{};
    p.f.feat = feat; p.f.frame_off = frame_off; p.f.whole = whole; p.f.n_utts = n_utts; p.f.n_feat = n_feat;
    p.f.win_len = win_len; p.f.shift_len = shift_len; p.f.spk_ptr = spk_ptr; p.f.spk_utts = spk_utts; p.f.n_spk = n_spk;
    p.f.stats = const_cast<float*>(stats);
    p.spk_of_utt = spk_of_utt;
    p.utt_ties = static_cast<int32_t*>(workspace);
    p.spk_ties = ties;
    SEPT_CUDA(sept::launch_speaker_stats_bwd_ties(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_speaker_stats_bwd_frames_f32(const float* feat, const int64_t* frame_off, const uint8_t* whole, int n_utts,
                                      int n_feat, int win_len, int shift_len, const int32_t* spk_of_utt,
                                      const float* stats, const float* dstats, const int32_t* ties, float* dfeat,
                                      sept_stream_t stream) {
    if (!feat || !frame_off || !spk_of_utt || !stats || !dstats || !ties || !dfeat || n_utts < 0 || n_feat <= 0 ||
        win_len <= 0 || shift_len <= 0)
        return fail(SEPT_E_BADARG, "sept_speaker_stats_bwd_frames_f32: bad argument");
    sept::SpeakerStatsBwdParams p{};
    p.f.feat = feat; p.f.frame_off = frame_off; p.f.whole = whole; p.f.n_utts = n_utts; p.f.n_feat = n_feat;
    p.f.win_len = win_len; p.f.shift_len = shift_len;
    p.f.stats = const_cast<float*>(stats);
    p.spk_of_utt = spk_of_utt; p.dstats = dstats; p.dfeat = dfeat;
    p.spk_ties = const_cast<int32_t*>(ties);                     // read only by the frames pass
    SEPT_CUDA(sept::launch_speaker_stats_bwd_frames(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_cloak_fwd_f32(const float* x, const float* locs, const float* rhos, const float* mask, const float* eps,
                       uint64_t seed, uint64_t offset, const uint64_t* draw_dev, int per_sample, float eps_std, float min_scale,
                       float max_scale, int batch, int wf, float* out, float* eps_out, float* noise_out, sept_stream_t stream) {
    if (!x || !locs || !rhos || !out || batch < 0 || wf <= 0) return fail(SEPT_E_BADARG, "sept_cloak_fwd_f32: bad argument");
    if (wf % 4) return fail(SEPT_E_BADARG, "sept_cloak_fwd_f32: W*F=%d must be a multiple of 4", wf);
    if (!aligned16(x) || !aligned16(locs) || !aligned16(rhos) || !aligned16(mask) || !aligned16(eps) || !aligned16(out) ||
        !aligned16(eps_out) || !aligned16(noise_out))
        return fail(SEPT_E_BADARG, "sept_cloak_fwd_f32: pointers must be 16-byte aligned");
    sept::CloakFwdParams p{};
    p.x = x; p.locs = locs; p.rhos = rhos; p.mask = mask; p.eps = eps; p.seed = seed; p.offset = offset; p.draw_dev = draw_dev; p.per_sample = per_sample ? 1 : 0;
    if (per_sample && noise_out) return fail(SEPT_E_BADARG, "sept_cloak_fwd_f32: noise_out is a single (wf) sample; not available with per_sample");
    p.eps_std = eps_std; p.min_scale = min_scale; p.max_scale = max_scale; p.batch = batch; p.wf = wf; p.out = out;
    p.eps_out = eps_out; p.noise_out = noise_out;
    SEPT_CUDA(sept::launch_cloak_fwd(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_counter_add_u64(uint64_t* counter_dev, uint64_t inc, sept_stream_t stream) {
    if (!counter_dev) return fail(SEPT_E_BADARG, "sept_counter_add_u64: null pointer");
    SEPT_CUDA(sept::launch_counter_add(counter_dev, inc, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_cloak_bwd_workspace_bytes(int wf) {
    if (wf <= 0) return 0;
    return (size_t)sept::kCloakSlices * wf * sizeof(float) + ((size_t)(wf + 511) / 512) * sizeof(unsigned) + 16;
}

int sept_cloak_grl_bwd_f32(const float* g_a, const float* g_b, float lambda, const float* eps, const float* rhos,
                           const float* mask, float min_scale, float max_scale, int batch, int wf, void* workspace,
                           float* dlocs, float* drhos, float* dx, sept_stream_t stream) {
    if (!g_a || !eps || !rhos || !workspace || !dlocs || batch < 0 || wf <= 0)
        return fail(SEPT_E_BADARG, "sept_cloak_grl_bwd_f32: bad argument");
    if (wf % 4) return fail(SEPT_E_BADARG, "sept_cloak_grl_bwd_f32: W*F=%d must be a multiple of 4", wf);
    if (!aligned16(g_a) || !aligned16(g_b) || !aligned16(eps) || !aligned16(rhos) || !aligned16(mask) ||
        !aligned16(workspace) || !aligned16(dlocs) || !aligned16(drhos) || !aligned16(dx))
        return fail(SEPT_E_BADARG, "sept_cloak_grl_bwd_f32: pointers must be 16-byte aligned");
    sept::CloakBwdParams p{};
    p.g_a = g_a; p.g_b = g_b; p.lambda = lambda; p.eps = eps; p.rhos = rhos; p.mask = mask;
    p.min_scale = min_scale; p.max_scale = max_scale; p.reg_coef = 0.f; p.batch = batch; p.wf = wf;
    p.partial = static_cast<float*>(workspace);
    p.counters = reinterpret_cast<unsigned*>(static_cast<float*>(workspace) + (size_t)sept::kCloakSlices * wf);
    p.dlocs = dlocs; p.drhos = drhos; p.dx = dx;
    SEPT_CUDA(sept::launch_cloak_bwd(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_grl_bwd_f32(const float* g, float lambda, int64_t n, float* dx, sept_stream_t stream) {
    if (n == 0) return SEPT_OK;
    if (!g || !dx || n < 0) return fail(SEPT_E_BADARG, "sept_grl_bwd_f32: bad argument");
    if (!aligned16(g) || !aligned16(dx)) return fail(SEPT_E_BADARG, "sept_grl_bwd_f32: pointers must be 16-byte aligned");
    SEPT_CUDA(sept::launch_grl_bwd(g, lambda, (size_t)n, dx, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_wave_cloak_layout(const int64_t* utt_off, int n_utts, int period, int64_t* tile_off) {
    if (!utt_off || !tile_off || n_utts < 0 || period <= 0) return fail(SEPT_E_BADARG, "sept_wave_cloak_layout: bad argument");
    if (period % 4) return fail(SEPT_E_BADARG, "sept_wave_cloak_layout: period=%d must be a multiple of 4", period);
    if (utt_off[0] < 0) return fail(SEPT_E_BADARG, "sept_wave_cloak_layout: utt_off[0] is negative");
    tile_off[0] = 0;
    for (int u = 0; u < n_utts; ++u) {
        const int64_t n = utt_off[u + 1] - utt_off[u];
        if (n < 0) return fail(SEPT_E_BADARG, "sept_wave_cloak_layout: offsets must be non-decreasing (utterance %d)", u);
        if (n >= (int64_t)1 << 31) return fail(SEPT_E_BADARG, "sept_wave_cloak_layout: utterance %d is longer than 2^31 samples", u);
        tile_off[u + 1] = tile_off[u] + (n + period - 1) / period;
    }
    return SEPT_OK;
}

int sept_wave_cloak_fwd_f32(const float* x, const int64_t* utt_off, int n_utts, int64_t n_samples, const float* noise,
                            int period, float* y, sept_stream_t stream) {
    if (!x || !utt_off || !noise || !y || n_utts < 0 || n_samples < 0 || period <= 0)
        return fail(SEPT_E_BADARG, "sept_wave_cloak_fwd_f32: bad argument");
    if (period % 4) return fail(SEPT_E_BADARG, "sept_wave_cloak_fwd_f32: period=%d must be a multiple of 4", period);
    if (!aligned16(x) || !aligned16(noise) || !aligned16(y))
        return fail(SEPT_E_BADARG, "sept_wave_cloak_fwd_f32: pointers must be 16-byte aligned");
    sept::WaveAddParams p{};
    p.x = x; p.utt_off = utt_off; p.n_utts = n_utts; p.n = n_samples; p.noise = noise; p.period = period; p.y = y;
    SEPT_CUDA(sept::launch_wave_add(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_wave_cloak_eval_workspace_bytes(int period) {
    return period > 0 && period % 4 == 0 ? (size_t)period * sizeof(float) : 0;
}

int sept_wave_cloak_eval_f32(const float* x, const int64_t* utt_off, int n_utts, int64_t n_samples, const float* locs,
                             const float* rhos, const float* eps, uint64_t seed, uint64_t offset, const uint64_t* draw_dev,
                             const int64_t* utt_draw_dev, float eps_std, float min_scale, float max_scale, int period,
                             void* workspace, float* y, sept_stream_t stream) {
    if (!x || !utt_off || !locs || !rhos || !workspace || !y || n_utts < 0 || n_samples < 0 || period <= 0)
        return fail(SEPT_E_BADARG, "sept_wave_cloak_eval_f32: bad argument");
    if (period % 4) return fail(SEPT_E_BADARG, "sept_wave_cloak_eval_f32: period=%d must be a multiple of 4", period);
    if (!aligned16(x) || !aligned16(locs) || !aligned16(rhos) || !aligned16(eps) || !aligned16(workspace) || !aligned16(y))
        return fail(SEPT_E_BADARG, "sept_wave_cloak_eval_f32: pointers must be 16-byte aligned");
    sept::WaveEvalParams p{};
    p.x = x; p.utt_off = utt_off; p.n_utts = n_utts; p.n = n_samples; p.locs = locs; p.rhos = rhos; p.eps = eps;
    p.seed = seed; p.offset = offset; p.draw = draw_dev; p.utt_draw = utt_draw_dev; p.eps_std = eps_std;
    p.min_scale = min_scale; p.max_scale = max_scale; p.period = period; p.sigma = static_cast<float*>(workspace); p.y = y;
    SEPT_CUDA(sept::launch_wave_eval(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_wave_cloak_bwd_workspace_bytes(int period) {
    return period > 0 && period % 4 == 0 ? (size_t)sept::kWaveSlices * period * sizeof(float) : 0;
}

int sept_wave_cloak_bwd_f32(const float* g, const int64_t* utt_off, const int64_t* tile_off, int n_utts, int64_t n_tiles,
                            int period, void* workspace, float* r, sept_stream_t stream) {
    if (!g || !utt_off || !tile_off || !workspace || !r || n_utts < 0 || n_tiles < 0 || period <= 0)
        return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_f32: bad argument");
    if (period % 4) return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_f32: period=%d must be a multiple of 4", period);
    if (!aligned16(g) || !aligned16(workspace) || !aligned16(r))
        return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_f32: pointers must be 16-byte aligned");
    sept::WaveReduceParams p{};
    p.g = g; p.utt_off = utt_off; p.tile_off = tile_off; p.n_utts = n_utts; p.n_tiles = n_tiles; p.period = period;
    p.partial = static_cast<float*>(workspace); p.r = r;
    SEPT_CUDA(sept::launch_wave_reduce(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

size_t sept_wave_cloak_bwd_per_utt_workspace_bytes(int period) {
    return period > 0 && period % 4 == 0 ? 2 * (size_t)sept::kWaveSlices * period * sizeof(float) : 0;
}

int sept_wave_cloak_bwd_per_utt_f32(const float* g, const int64_t* utt_off, const int64_t* tile_off, int n_utts,
                                    int64_t n_tiles, int period, const float* rhos, const float* eps, uint64_t seed,
                                    uint64_t offset, const uint64_t* draw_dev, const int64_t* utt_draw_dev, float eps_std,
                                    float min_scale, float max_scale, void* workspace, float* dlocs, float* drhos,
                                    sept_stream_t stream) {
    if (!g || !utt_off || !tile_off || !rhos || !workspace || !dlocs || !drhos || n_utts < 0 || n_tiles < 0 || period <= 0)
        return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_per_utt_f32: bad argument");
    if (period % 4) return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_per_utt_f32: period=%d must be a multiple of 4", period);
    if (!aligned16(g) || !aligned16(rhos) || !aligned16(eps) || !aligned16(workspace) || !aligned16(dlocs) || !aligned16(drhos))
        return fail(SEPT_E_BADARG, "sept_wave_cloak_bwd_per_utt_f32: pointers must be 16-byte aligned");
    sept::WaveReducePerUttParams p{};
    p.r.g = g; p.r.utt_off = utt_off; p.r.tile_off = tile_off; p.r.n_utts = n_utts; p.r.n_tiles = n_tiles;
    p.r.period = period; p.r.partial = static_cast<float*>(workspace); p.r.r = dlocs;
    p.rhos = rhos; p.eps = eps; p.seed = seed; p.offset = offset; p.draw = draw_dev; p.utt_draw = utt_draw_dev;
    p.eps_std = eps_std; p.min_scale = min_scale; p.max_scale = max_scale; p.drhos = drhos;
    SEPT_CUDA(sept::launch_wave_reduce_per_utt(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

int sept_add_noise_rows_f32(float* data_dev,const int64_t* job_row_dev, const int32_t* job_ptr_dev, const int64_t* draw_id_dev,
                            int n_jobs, int row_elems, uint64_t seed, float std, const float* noise_dev, sept_stream_t stream) {
    if (n_jobs == 0) return SEPT_OK;
    if (!data_dev || !job_row_dev || !job_ptr_dev || !draw_id_dev || n_jobs < 0 || row_elems <= 0)
        return fail(SEPT_E_BADARG, "sept_add_noise_rows_f32: bad argument");
    if (row_elems % 4 != 0) return fail(SEPT_E_UNSUPPORTED, "sept_add_noise_rows_f32: row_elems=%d must be a multiple of 4", row_elems);
    if (n_jobs > 65535) return fail(SEPT_E_UNSUPPORTED, "sept_add_noise_rows_f32: n_jobs=%d exceeds 65535 per call", n_jobs);
    if (!aligned16(data_dev) || (noise_dev && !aligned16(noise_dev)))
        return fail(SEPT_E_BADARG, "sept_add_noise_rows_f32: pointers must be 16-byte aligned");
    sept::AddNoiseParams p{};
    p.data = data_dev; p.job_row = job_row_dev; p.job_ptr = job_ptr_dev; p.draw_id = draw_id_dev; p.n_jobs = n_jobs;
    p.row_elems = row_elems; p.seed = seed; p.std = std; p.noise = noise_dev;
    SEPT_CUDA(sept::launch_add_noise(p, static_cast<cudaStream_t>(stream)));
    return SEPT_OK;
}

}  // extern "C"
