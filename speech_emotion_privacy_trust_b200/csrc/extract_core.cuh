// Per-lane phase functions of the fused frame -> window -> real FFT -> |X|^2 -> mel kernel.
//
// Work unit: one warp owns one ITEM = FPW consecutive frames of one utterance (FPW = 2 * 32/R: 8 / 4 / 2 frames
// for n_fft 400 / 800 / 1600) and takes it through every phase with only __syncwarp() in between, so the warps
// of an SM drift apart and the FP-heavy and the shared-memory-heavy phases of different warps overlap.
// Frames are processed in adjacent PAIRS packed into pk2 (vec.cuh).
//
// The functions are __host__ __device__ on purpose: the CUDA kernel (extract.cu) calls them with its lane id,
// and tests/hostsim calls the very same functions from a loop over lane ids with plain arrays standing in for
// shared memory, so the index algebra (prime-factor maps, real split, tile positions, reflect staging) is
// verified on a CPU-only box.  The host emulation is test code, not a fallback: the library has no CPU path.
//
// Warp-private shared memory (see DESIGN.md):
//   stage  float [2 + SPAN + 1], SPAN = (FPW-1)*hop + n_fft   reflect-padded waveform span of the item at offset 2,
//                                                one halo sample either side (for the waveform-gradient stream)
//   Y      pk2   [PPW][25 (+1) rows k2][re: R | im: R | pad 2]   pass 1 output / pass 2 input; each pk2 = (frame a, frame b);
//                                                the fused pass keeps a second copy of row 0 in row 25.
//                                                Real and imaginary parts sit in separate half rows so that their
//                                                8-byte stores cannot be fused into quads (which costs 4 MOVs each)
//   P      pk2   [PPW][PP] over the Y tile       4|X[k]|^2 of the frame pair at bin_pos(k) (written only after every Z
//                                                of the item has been read into registers), then three zero slots
// Replaces, for one item: torch.stft framing/window/rFFT + abs().pow(2) (torchaudio functional.py:123-144)
// and MelScale's matmul (transforms/_transforms.py:417).
#pragma once
#include "dft.cuh"
#ifdef __CUDACC__
#include "extract.h"
#endif

namespace sept {

struct alignas(8) f2 { float x, y; };
struct alignas(16) f4 { float x, y, z, w; };
struct alignas(16) pk4 { pk2 re, im; };

template <int R_>
struct Geo {
    static constexpr int R = R_;
    static constexpr int NC = R * 25, NFFT = 2 * NC, PAD = NFFT / 2;
    static constexpr int PPW = 32 / R;                           // packed frame pairs per warp
    static constexpr int FPW = 2 * PPW;                           // frames per item
    static constexpr int RS = 2 * R + 2;                          // pk2 per k2 row: [re: R][im: R][pad 2]; RS/2 odd spreads rows over banks
    static constexpr int YROWS = R <= 16 ? 26 : 25;               // fused pass: row 25 is a second copy of row 0 (see pass2_split)
    static constexpr int YP = YROWS * RS + 4;                     // pk2 per pair
    static constexpr int Y_PK2 = PPW * YP;                        // pk2 per warp
    static constexpr int Y_PK4 = Y_PK2 / 2;                       // the same in 16-byte units
    static constexpr int TWS = R + 1;                             // f2 per split-twiddle row (odd: rows spread over banks)
    static constexpr int PS_ROUNDS = (PPW + 1) / 2;               // fused pass-2 + split: lane = (pair p % 2, row pair j < 13)
    static constexpr int P2_TASKS = PPW * 25;                     // pass-2 row tasks per item
    static constexpr int LEAD = 2;                                // floats in front of the staged span (halo + 8-byte alignment)
    static SEPT_HD int span(int hop) { return (FPW - 1) * hop + NFFT; }
    // pk2 slot of bin k in a pair's power tile: natural order with gaps between blocks of bins, chosen per R so that
    // the 8-byte stores of the split (lanes = rows j of one k1 in the fused pass: bins 16 t + k1 of 13 different blocks
    // t; lanes = k1 in the R = 32 pass) spread over the 16 bank pairs.  Exhaustive search over k + ((c (k >> s)) >> d)
    // against the kernel's store pattern (tools/tile_layout_search.py): 76 / 80 wavefronts per item for R = 16 / 8 (64 is conflict free, the old
    // k + k/16 cost 128), and the plain order is conflict free for R = 32.  The mel gathers adapt through the table
    // scheduler (tables.h), so the layout is free to serve the stores.
    static constexpr SEPT_HD int bin_pos(int k) {
        return R == 32 ? k : R == 16 ? k + ((9 * (k >> 4)) >> 1) : k + ((9 * (k >> 3)) >> 2);
    }
    static constexpr int ZSLOT = bin_pos(NC) + 1, ZSLOTS = 3;     // kept at zero: idle slots of the mel program read them
    static constexpr int PP = (ZSLOT + ZSLOTS + 1) & ~1;          // pk2 per pair of the power tile (bins 0..NC, zero slots)
    static_assert(PPW * PP <= Y_PK2, "power tile must fit in the Y tile it overwrites");
    // fused pass 2 + split task of a lane in round r: pair p = 2r + lane/16, row pair j = lane%16 (idle when j >= 13)
    static SEPT_HD bool ps_task(int lane, int r, int& p, int& j) {
        p = 2 * r + (lane >> 4);
        j = lane & 15;
        return j < 13 && p < PPW;
    }
    static SEPT_HD int stage_floats(int hop) { return (LEAD + span(hop) + 1 + 3) & ~3; }
};

// ---- staging: reflect-padded span of the item starting at frame t0 ----------------------------------------
// padded index q = t0*hop + i maps to source sample q - pad, reflected without edge repeat
// (torch/functional.py:675-680).  deriv != 0 stages np.gradient(x) (audio_feature_extraction.py:20) instead.
SEPT_HD int reflect_src(long long q, int pad, int n) {
    long long s = q - pad;
    if (s < 0) s = -s;
    else if (s >= n) s = 2LL * (n - 1) - s;
    return (s >= 0 && s < n) ? (int)s : -1;
}

SEPT_HD float staged_sample(const float* wav, int n, int src, int deriv) {
    if (src < 0) return 0.f;
    if (!deriv) return wav[src];
    if (src == 0) return wav[1] - wav[0];
    if (src == n - 1) return wav[n - 1] - wav[n - 2];
    return (wav[src + 1] - wav[src - 1]) * 0.5f;
}

// generic staging (edge items: reflection, utterance ends, one-sided differences): stage[LEAD - 1 + i] = sample at
// padded index q0 - 1 + i, i = 0 .. span + 1.  Loads are issued in independent batches of 8 per lane.
template <class G>
SEPT_HD void stage_item(int lane, const float* wav, int n, int t0, int hop, int deriv, float* stage) {
    const long long q0 = (long long)t0 * hop - 1;
    const int count = G::span(hop) + 2;
    for (int base = 0; base < count; base += 256) {
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = base + j * 32 + lane;
            v[j] = i < count ? staged_sample(wav, n, reflect_src(q0 + i, G::PAD, n), deriv) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int i = base + j * 32 + lane;
            if (i < count) stage[G::LEAD - 1 + i] = v[j];
        }
    }
}

// true when the staged span (with its halo) of the item lies strictly inside the utterance: no reflection, no
// one-sided difference; such items are staged with asynchronous copies and differentiated in shared memory
template <class G>
SEPT_HD bool item_is_interior(int n, int t0, int hop) {
    const long long first = (long long)t0 * hop - G::PAD - 1;          // source index of the front halo
    return first >= 1 && first + G::span(hop) + 2 <= (long long)n - 1;
}

// ---- sources of the lane-constant tables.  The phase functions read the window and the split twiddles through one of
// these: from shared memory (generic kernel, host emulation) or from registers filled out of tensor memory (extract.cu) --
struct WinShared {                                               // win2[n] = (w[2n], w[2n+1])
    const f2* win2;
    SEPT_HD f2 at(int idx, int /*n2*/) const { return win2[idx]; }
};
struct TwShared {                                                // row of the lane: tws[j * TWS + k1]
    const f2* row;
    SEPT_HD f2 at(int k1) { return row[k1]; }
};

struct TwStrided {                                               // unfused pass (R = 32): the lane's twiddle of row k2
    const f2* col;                                               // tws + k1
    int stride;
    SEPT_HD f2 at(int k2) { return col[k2 * stride]; }
};

// ---- pass 1: lane (p, n1) windows the 25 complex samples z[n] = xw[2n] + i xw[2n+1], n = (25 n1 + R n2) mod NC,
// of frames 2p and 2p+1 and transforms them over n2 ------------------------------------------------------------
// DIFF: the stage holds the raw waveform of an interior item and the stream wanted is np.gradient of it
// (audio_feature_extraction.py:20): the central difference (x[j+1] - x[j-1]) / 2 is taken on the fly from the
// neighbouring sample pairs, the 1/2 riding on the window (exact: a power of two).
template <class G, bool DIFF, class Win>
SEPT_HD void pass1_load(int lane, const float* stage, int hop, const Win& win, pk2 (&re)[25], pk2 (&im)[25]) {
    constexpr int R = G::R;
    const int p = lane / R, n1 = lane % R;
    const f2* xa = reinterpret_cast<const f2*>(stage + G::LEAD + (2 * p) * hop);
    const f2* xb = reinterpret_cast<const f2*>(stage + G::LEAD + (2 * p + 1) * hop);
#pragma unroll
    for (int n2 = 0; n2 < 25; ++n2) {
        const int idx = Pfa<R>::in_index(n1, n2);
        const f2 w = win.at(idx, n2);
        if (!DIFF) {
            const f2 a = xa[idx], b = xb[idx];
            re[n2] = pk(a.x * w.x, b.x * w.x);
            im[n2] = pk(a.y * w.y, b.y * w.y);
        } else {
            const f2 al = xa[idx - 1], a = xa[idx], ar = xa[idx + 1];
            const f2 bl = xb[idx - 1], b = xb[idx], br = xb[idx + 1];
            const float hx = 0.5f * w.x, hy = 0.5f * w.y;
            re[n2] = pk((a.y - al.y) * hx, (b.y - bl.y) * hx);
            im[n2] = pk((ar.x - a.x) * hy, (br.x - b.x) * hy);
        }
    }
}

template <class G>
SEPT_HD void pass1_transform_store(int lane, pk2 (&re)[25], pk2 (&im)[25], pk2* Y) {
    constexpr int R = G::R;
    const int p = lane / R, n1 = lane % R;
    Dft<25>::run(re, im);
    pk2* y = Y + p * G::YP + n1;
#pragma unroll
    for (int k2 = 0; k2 < 25; ++k2) { y[k2 * G::RS] = re[k2]; y[k2 * G::RS + R] = im[k2]; }
    // the fused pass reads row 0 as its own partner; a second copy in row 25 keeps that 16-byte read out of the bank
    // group of row 24 (rows 0 and 24 are 24 * RS * 8 bytes = a multiple of 128 apart)
    if (G::YROWS == 26) { y[25 * G::RS] = re[0]; y[25 * G::RS + R] = im[0]; }
}

// Two forms of the same pass.  pass1<G, DIFF>: loads and transform are one straight-line block per stream kind (the loads
// overlap the first butterflies).  pass1_shared<G>: only the LOADS differ between the two streams (run-time, warp-uniform
// `diff`), the 25-point transform behind them exists once -- so both MFCC streams of an item run through the same code.
// Which one a kernel uses is decided by its instruction-cache footprint (extract.cu: kSharedPass1).
template <class G, bool DIFF, class Win>
SEPT_HD void pass1(int lane, const float* stage, int hop, const Win& win, pk2* Y) {
    pk2 re[25], im[25];
    pass1_load<G, DIFF>(lane, stage, hop, win, re, im);
    pass1_transform_store<G>(lane, re, im, Y);
}

template <class G, class Win>
SEPT_HD void pass1_shared(int lane, const float* stage, int hop, const Win& win, pk2* Y, bool diff) {
    pk2 re[25], im[25];
    if (!diff) pass1_load<G, false>(lane, stage, hop, win, re, im);
    else pass1_load<G, true>(lane, stage, hop, win, re, im);
    pass1_transform_store<G>(lane, re, im, Y);
}

// load one k2 row (R complex samples of a frame pair) with 16-byte loads of two neighbouring real / imaginary parts
template <int R>
SEPT_HD void load_row(const pk2* y, pk2 (&re)[R], pk2 (&im)[R]) {
#pragma unroll
    for (int i = 0; i < R; i += 2) {
        const pk4 a = *reinterpret_cast<const pk4*>(y + i);
        const pk4 b = *reinterpret_cast<const pk4*>(y + R + i);
        re[i] = a.re; re[i + 1] = a.im;                          // pk4's two halves: elements i and i+1
        im[i] = b.re; im[i + 1] = b.im;
    }
}

// ---- pass 2 (unfused form, R = 32): row task (p, k2) transforms its R samples over n1, in place ----------------
template <class G>
SEPT_HD void pass2_row(int task, pk2* Y) {
    constexpr int R = G::R;
    const int p = task / 25, k2 = task % 25;
    pk2* y = Y + p * G::YP + k2 * G::RS;
    pk2 re[R], im[R];
    load_row<R>(y, re, im);
    Dft<R>::run(re, im);
#pragma unroll
    for (int i = 0; i < R; ++i) { y[i] = re[i]; y[R + i] = im[i]; }
}

// ---- real split of one conjugate pair: Zk = Z[k], Zm = Z[NC-k], tw = W_{NFFT}^k.  Returns 4|X[k]|^2 and
// 4|X[NC-k]|^2 (the 1/4 is folded into the mel weights).  X[k] = E + W^k O with E = (Zk + conj Zm)/2,
// O = (Zk - conj Zm)/(2i); X[NC-k] = conj(E - W^k O). ------------------------------------------------------
SEPT_HD void split_pair(pk4 zk, pk4 zm, pk2 twr, pk2 twi, pk2& pk_, pk2& pm_) {
    const pk2 er = zk.re + zm.re, ei = zk.im - zm.im;
    const pk2 o_r = zk.im + zm.im, o_i = zm.re - zk.re;          // (Zk - conj Zm) / i
    const pk2 tr = fnma2(o_i, twi, o_r * twr), ti = fma2(o_i, twr, o_r * twi);
    const pk2 xr = er + tr, xi = ei + ti, yr = er - tr, yi = ei - ti;
    pk_ = fma2(xi, xi, xr * xr);
    pm_ = fma2(yi, yi, yr * yr);
}

// iteration k2 (0..12) of the split: lane (p, k1) pairs Z at (k1, k2) with Z at (R-k1, 25-k2).
// Returns false when the lane has nothing to do (row 0 is its own partner: only k1 <= R/2 work).
template <class G, class Tw>
SEPT_HD bool split_load(int lane, int k2, const pk2* Y, Tw& tws, pk2& pk_, pk2& pm_) {
    constexpr int R = G::R;
    const int p = lane / R, k1 = lane % R, km = (R - k1) % R;
    const f2 tw = tws.at(k2);                                     // the lane's twiddle of row k2; fetched by every lane (warp-wide source)
    if (k2 == 0 && k1 > R / 2) return false;
    const int rb = (25 - k2) % 25;
    const pk2* yk = Y + p * G::YP + k2 * G::RS + k1;
    const pk2* ym = Y + p * G::YP + rb * G::RS + km;
    const pk4 zk{yk[0], yk[R]}, zm{ym[0], ym[R]};
    split_pair(zk, zm, splat(tw.x), splat(tw.y), pk_, pm_);
    return true;
}

// ---- fused pass 2 + split (R <= 16): task (p, j) transforms rows j and 25-j of pair p over n1 in registers and
// splits them against each other without another trip through shared memory.  pu[k1] = 4|X|^2 at bin CRT(k1, j),
// pv[k1] = 4|X|^2 at bin CRT(k1, 25-j).  Row 0 (j = 0) is its own partner: pu holds the whole row and pv[0] the
// Nyquist bin. ------------------------------------------------------------------------------------------------------
template <class G, class Tw>
SEPT_HD void pass2_split(int p, int j, const pk2* Y, Tw& tw, pk2 (&pu)[G::R], pk2 (&pv)[G::R]) {
    constexpr int R = G::R;
    const int rb = 25 - j;                                        // j = 0: row 25, the copy of row 0
    pk2 ur[R], ui[R], vr[R], vi[R];
    load_row<R>(Y + p * G::YP + j * G::RS, ur, ui);
    load_row<R>(Y + p * G::YP + rb * G::RS, vr, vi);
    Dft<R>::run(ur, ui);
    Dft<R>::run(vr, vi);
#pragma unroll
    for (int k1 = 0; k1 < R; ++k1) {
        const int km = (R - k1) % R;
        const f2 w = tw.at(k1);
        split_pair(pk4{ur[k1], ui[k1]}, pk4{vr[km], vi[km]}, splat(w.x), splat(w.y), pu[k1], pv[km]);
    }
}

template <class G>
SEPT_HD void pass2_split_store(int p, int j, pk2* P, const pk2 (&pu)[G::R], const pk2 (&pv)[G::R]) {
    constexpr int R = G::R, NC = G::NC;
    const int rb = (25 - j) % 25;
    pk2* base = P + p * G::PP;
    const int kj = (Pfa<R>::cK2 * j) % NC, kb = (Pfa<R>::cK2 * rb) % NC;
#pragma unroll
    for (int k1 = 0; k1 < R; ++k1) {
        const int c1 = (Pfa<R>::cK1 * k1) % NC;                  // compile-time after unrolling
        int k = kj + c1;
        if (k >= NC) k -= NC;
        base[G::bin_pos(k)] = pu[k1];
        if (j > 0) {
            int kk = kb + c1;
            if (kk >= NC) kk -= NC;
            base[G::bin_pos(kk)] = pv[k1];
        }
    }
    if (j == 0) {
        base[G::bin_pos(NC)] = pv[0];
#pragma unroll
        for (int z = 0; z < G::ZSLOTS; ++z) base[G::ZSLOT + z] = splat(0.f);
    }
}

// after EVERY lane holds its 13 conjugate pairs in registers (warp barrier), the Y tile is overwritten by the power
// tile: lane (p, k1) stores bins k = CRT(k1, k2) (k mod R = k1, k mod 25 = k2) and NC - k for k2 = 0..12.  Consecutive
// lanes hit consecutive residues mod R, so the 8-byte stores are bank-conflict free.
template <class G>
SEPT_HD void split_store_all(int lane, pk2* P, const pk2 (&a)[13], const pk2 (&b)[13], bool on0) {
    constexpr int R = G::R;
    int k = (Pfa<R>::cK1 * (lane % R)) % G::NC;                  // CRT(k1, 0); + cK2 per k2 step
    pk2* base = P + (lane / R) * G::PP;
#pragma unroll
    for (int k2 = 0; k2 <= 12; ++k2) {
        if (k2 > 0 || on0) {
            base[G::bin_pos(k)] = a[k2];
            if (k != G::NC - k) base[G::bin_pos(G::NC - k)] = b[k2];   // k = 0 pairs with the Nyquist bin NC; NC/2 is its own partner
            if (k == 0) {
#pragma unroll
                for (int z = 0; z < G::ZSLOTS; ++z) base[G::ZSLOT + z] = splat(0.f);
            }
        }
        k += Pfa<R>::cK2;
        if (k >= G::NC) k -= G::NC;
    }
}

// ---- mel: one round of the gather program (tables.h: make_mel_program) for one lane.  The lane's interval i yields
// U = sum of rising weights x power (band i) and D = sum of falling weights x power (band i-1) for every frame pair of
// the item; e points at the lane's entry of the round's first step, entries of one step are `width` apart.  Replaces
// MelScale's matmul (_transforms.py:417) -------------------------------------------------------------------------------
struct alignas(16) mel_step { float up, dn; int off, pad; };

template <class G>
SEPT_HD void mel_round(const pk2* P, const mel_step* e, int n_steps, int width, pk2 (&U)[G::PPW], pk2 (&D)[G::PPW]) {
#pragma unroll
    for (int p = 0; p < G::PPW; ++p) { U[p] = splat(0.f); D[p] = splat(0.f); }
    const unsigned char* base = reinterpret_cast<const unsigned char*>(P);
#pragma unroll 2
    for (int s = 0; s < n_steps; ++s) {
        const mel_step st = e[s * width];
        const pk2 up = splat(st.up), dn = splat(st.dn);
#pragma unroll
        for (int p = 0; p < G::PPW; ++p) {
            const pk2 v = *reinterpret_cast<const pk2*>(base + st.off + p * (G::PP * 8));
            U[p] = fma2(v, up, U[p]);
            D[p] = fma2(v, dn, D[p]);
        }
    }
}

// step counts of the reference's only filterbank (128 HTK mels, 16 kHz; audio_feature_extraction.py:36,42 and the
// MFCC melkwargs): head entries, then the four rounds.  The library compares them with the program it builds and
// falls back to the table-driven loops when they differ.
template <int R> struct FastMel;
template <> struct FastMel<8> { static constexpr int head = 0, s0 = 1, s1 = 2, s2 = 2, s3 = 5; };
template <> struct FastMel<16> { static constexpr int head = 0, s0 = 2, s1 = 3, s2 = 5, s3 = 9; };
template <> struct FastMel<32> { static constexpr int head = 1, s0 = 3, s1 = 5, s2 = 9, s3 = 17; };

// interval 0 (bins below the first mel point): rising side of band 0, the same for every lane (broadcast reads)
template <class G>
SEPT_HD void mel_head(const pk2* P, const mel_step* head, int n_head, pk2 (&U)[G::PPW]) {
#pragma unroll
    for (int p = 0; p < G::PPW; ++p) U[p] = splat(0.f);
    const unsigned char* base = reinterpret_cast<const unsigned char*>(P);
    for (int s = 0; s < n_head; ++s) {
        const mel_step st = head[s];
#pragma unroll
        for (int p = 0; p < G::PPW; ++p)
            U[p] = fma2(*reinterpret_cast<const pk2*>(base + st.off + p * (G::PP * 8)), splat(st.up), U[p]);
    }
}

// true when the program has the step counts of FastMel<R>: the forward then runs its unrolled path, which takes the
// falling weight as 1/4 - rising, and the backward must do the same to recompute the forward's mel power
template <int R>
inline bool fast_ok(int n_head, const int* st) {
    using F = FastMel<R>;
    return n_head == F::head && st[0] == F::s0 && st[1] == F::s1 && st[2] == F::s2 && st[3] == F::s3;
}

inline bool extract_mel_fast_ok(int n_fft, int n_mels, int n_head, const int* round_steps, int n_rounds) {
    if (n_mels != 128 || n_rounds != 4) return false;
    switch (n_fft) {
        case 400: return fast_ok<8>(n_head, round_steps);
        case 800: return fast_ok<16>(n_head, round_steps);
        case 1600: return fast_ok<32>(n_head, round_steps);
    }
    return false;
}

// ---- CTA-shared constants of the extraction kernel and its backward, in front of the warp tiles: mel gather program
// [n_mel_entries], window [NC] f2, split twiddles [13][R + 1] f2
SEPT_HD int extract_const_bytes(int R, int n_mel_entries) {
    return (n_mel_entries * 16 + R * 25 * 8 + 13 * (R + 1) * 8 + 15) & ~15;
}

#ifdef __CUDACC__
struct CtaConsts {
    mel_step* mel;
    f2* win2;
    f2* tws;
};

// thread tid of the CTA's n_threads copies its share of the constants of prm to the front of shared memory; a
// __syncthreads() must precede any read.  The kernel passes threadIdx.x and blockDim.x: read there, they carry the
// ranges of its launch bounds, which spare the loops a guard.
template <class G>
__device__ __forceinline__ CtaConsts load_cta_consts(unsigned tid, unsigned n_threads, unsigned char* smem,
                                                     const ExtractParams& prm) {
    CtaConsts c;
    c.mel = reinterpret_cast<mel_step*>(smem);
    c.win2 = reinterpret_cast<f2*>(c.mel + prm.n_mel_entries);
    c.tws = c.win2 + G::NC;
    for (int i = tid; i < 13 * G::TWS; i += n_threads) c.tws[i] = reinterpret_cast<const f2*>(prm.tws)[i];
    for (int i = tid; i < prm.n_mel_entries; i += n_threads)
        reinterpret_cast<f4*>(c.mel)[i] = reinterpret_cast<const f4*>(prm.mel_prog)[i];
    for (int i = tid; i < G::NC; i += n_threads) c.win2[i] = reinterpret_cast<const f2*>(prm.window)[i];
    return c;
}

// utterance u with off[u] <= x < off[u + 1] (off: item or sample offsets)
template <class Off, class Key>
__device__ __forceinline__ int find_utt(const Off* off, int n_utts, Key x) {
    int lo_ = 0, hi_ = n_utts - 1;
    while (lo_ < hi_) {
        const int mid = (lo_ + hi_) >> 1;
        if (__ldg(off + mid + 1) > x) hi_ = mid; else lo_ = mid + 1;
    }
    return lo_;
}
#endif

}  // namespace sept
