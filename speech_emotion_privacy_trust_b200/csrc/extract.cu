// Fused speech feature extraction kernels for sm_100a (see extract_core.cuh for the per-lane phases).
//
//   extract_kernel<R, MODE, FAST>  persistent, one CTA per SM; each WARP walks its share of the items (an item = FPW
//                             consecutive frames of one utterance) through stage -> window+DFT25 -> DFT-R ->
//                             real split+power -> mel gather program -> log, touching HBM only for the waveform span
//                             and the finished features.  FAST (the reference's 128-band filterbank): the lane-constant
//                             tables -- window samples, split twiddles, mel program -- live in tensor memory (tmem.cuh)
//                             and the mel phase is unrolled; otherwise they are read from shared memory.
//   (the second phase of MFCC -- per-utterance top_db floor + ortho DCT-II -- lives in mfcc_dct.cu)
//
// Replaces torchaudio MelSpectrogram/AmplitudeToDB/MFCC as called by
// feature_extraction/audio_feature_extraction.py:15-46 of the reference.
#include <cuda_runtime.h>
#include <cstdint>
#include <type_traits>

#include "extract.h"
#include "extract_core.cuh"
#include "tmem.cuh"

namespace sept {

constexpr float kDbPerLog2 = 3.01029995663981195f;   // 10*log10(2)
constexpr float kAmin = 1e-10f;                        // amplitude_to_DB amin (functional.py:390)

// 10*log10(max(p, 1e-10)) through MUFU.LG2 (abs. error ~1e-6 in log2 => ~1e-5 dB); the clamp keeps the argument normal,
// so the flush-to-zero form needs no denormal branch
__device__ __forceinline__ float power_to_db(float p) {
    float l;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(fmaxf(p, kAmin)));
    return kDbPerLog2 * l;
}

// ---- asynchronous staging (LDGSTS): the next item's waveform span lands in shared memory while the current item is
// still in its shared-memory phases ----------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async_f32(float* smem_dst, const float* gmem_src) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

struct ItemRef {
    const float* wav;      // utterance start
    long long f0;          // first output frame of the utterance
    int n, T, t0, u;
    bool interior;
};

struct MelJob {
    long long f0;          // first output frame of the utterance
    int T, t0, u, stream;  // frames of the utterance, first frame of the item, utterance, MFCC stream
};

// mel bands of every frame pair of one item: gather program over the power tile (lane = interval, see tables.h), hand
// the rising sums to the next band, log, store; lane = band in the stores.  Every lane runs every round (the step count
// is warp uniform).
template <class G, int MODE>
__device__ __forceinline__ void mel_rounds(int lane, const pk2* P, const mel_step* prog, int n_mels,
                                           const ExtractParams& prm, const MelJob& job) {
    float vmax = 0.f;
    const int width = n_mels < 32 ? n_mels : 32;
    const mel_step* e = prog + prm.n_mel_head + (lane < width ? lane : width - 1);
    pk2 carry[G::PPW];                                            // rising sum of the interval below the round's first
    mel_head<G>(P, prog, prm.n_mel_head, carry);
    for (int m0 = 0; m0 < n_mels; m0 += 32) {
        const int m = m0 + lane < n_mels ? m0 + lane : n_mels - 1;
        const bool live = m0 + lane < n_mels;
        const int n_steps = __shfl_sync(0xffffffffu, e->pad, 0);  // the round's first step carries its step count
        pk2 U[G::PPW], D[G::PPW];
        mel_round<G>(P, e, n_steps, width, U, D);
        e += n_steps * width;
#pragma unroll
        for (int p = 0; p < G::PPW; ++p) {
            pk2 below = shfl_up(U[p], 1);
            if (lane == 0) below = carry[p];
            carry[p] = shfl_lane(U[p], 31);
            const pk2 acc = below + D[p];
            const int ta = live ? job.t0 + 2 * p : job.T;         // lanes past the last band store nothing
            const float va = lo(acc), vb = hi(acc);
            if (MODE == kModeDbFrameMajor) {
                float* o = prm.out + (job.f0 + ta) * n_mels + m;
                if (ta < job.T) o[0] = power_to_db(va);
                if (ta + 1 < job.T) o[n_mels] = power_to_db(vb);
            } else if (MODE == kModeDbBandMajor) {
                float* o = prm.out + job.f0 * n_mels + (long long)m * job.T + ta;
                if (ta < job.T) o[0] = power_to_db(va);
                if (ta + 1 < job.T) o[1] = power_to_db(vb);
            } else {                                              // raw mel power, frame major, per stream
                float* o = prm.out + ((long long)job.stream * prm.total_frames + job.f0 + ta) * n_mels + m;
                if (ta < job.T) { o[0] = va; vmax = fmaxf(vmax, va); }
                if (ta + 1 < job.T) { o[n_mels] = vb; vmax = fmaxf(vmax, vb); }
            }
        }
    }
    if (MODE == kModeMfccPower) {
        if (job.stream == 0 && lane < G::FPW && job.t0 + lane < job.T)
            prm.frame_utt[job.f0 + job.t0 + lane] = job.u;        // saves the DCT kernel a search per frame
        // per-utterance max of the mel power (top_db floor, functional.py:393-402); non-negative floats order like
        // their bit patterns
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
        if (lane == 0) atomicMax(prm.utt_max + (long long)job.stream * prm.n_utts + job.u, __float_as_int(vmax));
    }
}

// ---- the compiled-in 128-band program (FastMel<R>) from tensor memory -----------------------------------------------
// TMEM columns of a lane: [0, 2 n) = {rising weight, byte offset} of its n = head + s0 + s1 + s2 + s3 program entries
// (the falling weight of a bin is 1/4 minus its rising weight: the triangles of neighbouring bands sum to one).
template <int R> struct TmemMap {
    using F = FastMel<R>;
    static constexpr int kMelEntries = F::head + F::s0 + F::s1 + F::s2 + F::s3;
    static constexpr int kTwEntries = R <= 16 ? R : 16;          // fused pass: W^k of the lane's row j for k1 < R; R = 32: rows k2 <= 12 of column k1
    static constexpr int kMel = 0, kTw = 2 * kMelEntries, kWin = kTw + 2 * kTwEntries, kEnd = kWin + 50;
    static constexpr uint32_t kCols = kEnd <= 32 ? 32 : kEnd <= 64 ? 64 : kEnd <= 128 ? 128 : 256;
};

// the lane's 25 window pairs (w[2n], w[2n+1]) in n2 order, in registers for the whole of pass 1
struct WinRegs {
    uint32_t w[50];
    __device__ __forceinline__ void load(uint32_t addr) { tmem::ld<50>(addr, w); tmem::wait_ld(); }
    __device__ __forceinline__ f2 at(int /*idx*/, int n2) const { return f2{__uint_as_float(w[2 * n2]), __uint_as_float(w[2 * n2 + 1])}; }
};

// the lane's split twiddles, fetched four at a time while the split walks over them (k is a compile-time constant at
// every call site, so the fetches sit at fixed places in the unrolled code; every lane of the warp must call)
struct TwTmem {
    uint32_t addr;
    uint32_t buf[8];
    __device__ __forceinline__ f2 at(int k) {
        if (k % 4 == 0) { tmem::ld<8>(addr + 2 * k, buf); tmem::wait_ld(); }
        return f2{__uint_as_float(buf[2 * (k % 4)]), __uint_as_float(buf[2 * (k % 4) + 1])};
    }
};

// one round of N steps whose entries sit in registers mp[2 s] = rising weight, mp[2 s + 1] = byte offset
template <class G, int N>
__device__ __forceinline__ void mel_round_regs(const pk2* P, const uint32_t* mp, pk2 (&U)[G::PPW], pk2 (&D)[G::PPW]) {
    const unsigned char* base = reinterpret_cast<const unsigned char*>(P);
#pragma unroll
    for (int p = 0; p < G::PPW; ++p) { U[p] = splat(0.f); D[p] = splat(0.f); }
#pragma unroll
    for (int s = 0; s < N; ++s) {
        const float upw = __uint_as_float(mp[2 * s]);
        const pk2 up = splat(upw), dn = splat(0.25f - upw);
#pragma unroll
        for (int p = 0; p < G::PPW; ++p) {
            const pk2 v = *reinterpret_cast<const pk2*>(base + mp[2 * s + 1] + p * (G::PP * 8));
            U[p] = fma2(v, up, U[p]);
            D[p] = fma2(v, dn, D[p]);
        }
    }
}

// fill the calling warp's TMEM quarter with its lanes' program (every warp does; warps w and w + 4 write the same values)
template <class G>
__device__ __forceinline__ void tmem_fill_mel(uint32_t taddr, int lane, const mel_step* prog) {
    using F = FastMel<G::R>;
    using M = TmemMap<G::R>;
    uint32_t v[2 * M::kMelEntries];
#pragma unroll
    for (int s = 0; s < M::kMelEntries; ++s) {
        const mel_step st = s < F::head ? prog[s] : prog[F::head + (s - F::head) * 32 + lane];
        v[2 * s] = __float_as_uint(st.up);
        v[2 * s + 1] = (uint32_t)st.off;
    }
    tmem::st<2 * M::kMelEntries>(taddr + M::kMel, v);
}

// ... and with its window samples (n2 order of pass 1) and split twiddles
template <class G>
__device__ __forceinline__ void tmem_fill_fft(uint32_t taddr, int lane, const f2* win2, const f2* tws) {
    using M = TmemMap<G::R>;
    constexpr int R = G::R;
    {
        uint32_t v[50];
#pragma unroll
        for (int n2 = 0; n2 < 25; ++n2) {
            const f2 w = win2[Pfa<R>::in_index(lane % R, n2)];
            v[2 * n2] = __float_as_uint(w.x);
            v[2 * n2 + 1] = __float_as_uint(w.y);
        }
        tmem::st<50>(taddr + M::kWin, v);
    }
    {
        uint32_t v[2 * M::kTwEntries];
#pragma unroll
        for (int k = 0; k < M::kTwEntries; ++k) {
            f2 w{0.f, 0.f};
            if (R <= 16) { const int j = (lane & 15) < 13 ? (lane & 15) : 12; w = tws[j * G::TWS + k]; }
            else if (k <= 12) w = tws[k * G::TWS + lane];
            v[2 * k] = __float_as_uint(w.x);
            v[2 * k + 1] = __float_as_uint(w.y);
        }
        tmem::st<2 * M::kTwEntries>(taddr + M::kTw, v);
    }
}

// mel bands, log, store of one item: no loops, no table reads from shared memory, one 64-bit address per item with
// immediate offsets for the stores
template <class G, int MODE>
__device__ __forceinline__ void mel_fast(int lane, const pk2* P, uint32_t taddr, const ExtractParams& prm, const MelJob& job) {
    using F = FastMel<G::R>;
    using M = TmemMap<G::R>;
    constexpr int PPW = G::PPW;
    uint32_t mp[2 * M::kMelEntries];
    tmem::ld<2 * M::kMelEntries>(taddr + M::kMel, mp);
    tmem::wait_ld();
    pk2 U[4][PPW], D[4][PPW], carry[PPW];
#pragma unroll
    for (int p = 0; p < PPW; ++p) carry[p] = splat(0.f);
#pragma unroll
    for (int s = 0; s < F::head; ++s)                              // interval 0: the same entries in every lane
#pragma unroll
        for (int p = 0; p < PPW; ++p)
            carry[p] = fma2(*reinterpret_cast<const pk2*>(reinterpret_cast<const unsigned char*>(P) + mp[2 * s + 1] + p * (G::PP * 8)),
                            splat(__uint_as_float(mp[2 * s])), carry[p]);
    const uint32_t* e = mp + 2 * F::head;
    mel_round_regs<G, F::s0>(P, e, U[0], D[0]);
    mel_round_regs<G, F::s1>(P, e + 2 * F::s0, U[1], D[1]);
    mel_round_regs<G, F::s2>(P, e + 2 * (F::s0 + F::s1), U[2], D[2]);
    mel_round_regs<G, F::s3>(P, e + 2 * (F::s0 + F::s1 + F::s2), U[3], D[3]);
    const int left = job.T - job.t0;                              // frames of the utterance from the item's first on
    float* o;
    if (MODE == kModeDbBandMajor) o = prm.out + job.f0 * 128 + (long long)lane * job.T + job.t0;
    else o = prm.out + ((MODE == kModeMfccPower ? (long long)job.stream * prm.total_frames : 0) + job.f0 + job.t0) * 128 + lane;
    const int band_stride = 32 * job.T;
    float vmax = 0.f;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
        for (int p = 0; p < PPW; ++p) {
            pk2 below = shfl_up(U[r][p], 1);
            if (r > 0) carry[p] = shfl_lane(U[r - 1][p], 31);    // every lane takes part in the shuffle
            if (lane == 0) below = carry[p];
            const pk2 acc = below + D[r][p];
            float va = lo(acc), vb = hi(acc);
            if (MODE == kModeMfccPower) { if (2 * p < left) vmax = fmaxf(vmax, va); if (2 * p + 1 < left) vmax = fmaxf(vmax, vb); }
            else { va = power_to_db(va); vb = power_to_db(vb); }
            if (MODE == kModeDbBandMajor) {
                if (2 * p < left) o[r * band_stride + 2 * p] = va;
                if (2 * p + 1 < left) o[r * band_stride + 2 * p + 1] = vb;
            } else {
                if (2 * p < left) o[(2 * p) * 128 + 32 * r] = va;
                if (2 * p + 1 < left) o[(2 * p + 1) * 128 + 32 * r] = vb;
            }
        }
    }
    if (MODE == kModeMfccPower) {
        if (job.stream == 0 && lane < G::FPW && lane < left) prm.frame_utt[job.f0 + job.t0 + lane] = job.u;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, d));
        if (lane == 0) atomicMax(prm.utt_max + (long long)job.stream * prm.n_utts + job.u, __float_as_int(vmax));
    }
}

template <int R, int MODE, bool FAST>
__global__ void __launch_bounds__(ExtractWarps<R>::value * 32, 1) extract_kernel(const ExtractParams prm) {
    using G = Geo<R>;
    const int kExtractWarps = blockDim.x >> 5;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int hop = prm.hop, n_mels = prm.n_mels;
    const int stage_floats = G::stage_floats(hop);

    const CtaConsts cc = load_cta_consts<G>(threadIdx.x, blockDim.x, smem_raw, prm);
    mel_step* melp = cc.mel;
    f2* win2 = cc.win2;
    f2* tws = cc.tws;
    uint32_t taddr = 0;                                           // this warp's quarter of the CTA's tensor memory
    __shared__ uint32_t tmem_base;
    // ---- this CTA's contiguous item range.  kDynamicItems: its warps draw items from a shared counter instead of
    // interleaving statically, so a warp that met edge items (reflection, utterance ends) does not hold the others up:
    // MFCC 4.04 -> 3.92 ms, n_fft 1600 7.04 -> 6.94 ms per corpus; the n_fft 800 dB kernel LOSES 3 % with it and keeps
    // the static interleave (A/B inside single runs, profiles/ab_dynamic_r02.log).  These kernels are sensitive to code
    // layout at the +-2 % level (80 KB of straight-line code against the instruction cache): the range is computed early
    // for the dynamic kernels and where it always was for the static one, which keeps the n_fft 800 kernel's SASS
    // byte-identical to the measured one.
    constexpr bool kDynamicItems = !(R == 16 && MODE != kModeMfccPower);
    __shared__ int cta_next;
    int n_items = 0, begin = 0, end = 0;
    if constexpr (kDynamicItems) {
        n_items = __ldg(prm.item_off + prm.n_utts);
        begin = (int)((long long)n_items * blockIdx.x / gridDim.x);
        end = (int)((long long)n_items * (blockIdx.x + 1) / gridDim.x);
        if (threadIdx.x == 0) cta_next = begin;
    }
    if constexpr (FAST) {
        if (warp == 0) tmem::alloc(&tmem_base, TmemMap<R>::kCols);
        tmem::fence_before_sync();
        __syncthreads();
        tmem::fence_after_sync();
        taddr = tmem::quarter_addr(tmem_base, warp, 0);
        tmem_fill_mel<G>(taddr, lane, melp);
        tmem_fill_fft<G>(taddr, lane, win2, tws);
        tmem::wait_st();
        tmem::fence_before_sync();
    }
    __syncthreads();
    if constexpr (FAST) tmem::fence_after_sync();

    // ---- warp-private tiles -------------------------------------------------------------------------------
    const int warp_bytes = stage_floats * 4 + G::Y_PK4 * 16;
    unsigned char* wbase = smem_raw + extract_const_bytes(R, prm.n_mel_entries) + warp * warp_bytes;
    float* stage = reinterpret_cast<float*>(wbase);
    pk2* Y = reinterpret_cast<pk2*>(wbase + stage_floats * 4);
    pk2* P = Y;

    if constexpr (!kDynamicItems) {
        n_items = __ldg(prm.item_off + prm.n_utts);
        begin = (int)((long long)n_items * blockIdx.x / gridDim.x);
        end = (int)((long long)n_items * (blockIdx.x + 1) / gridDim.x);
    }
    auto grab = [&]() {                                           // next item of the CTA (>= end: none left); ascending per warp
        int v = 0;
        if (lane == 0) v = atomicAdd(&cta_next, 1);
        return __shfl_sync(0xffffffffu, v, 0);
    };
    int item;
    if constexpr (kDynamicItems) item = grab();
    else item = begin + warp;
    const bool active = item < end;                               // idle warps still reach the barrier at the end
    int u = active ? find_utt(prm.item_off, prm.n_utts, item) : 0;
    int u_first = __ldg(prm.item_off + u), u_last = __ldg(prm.item_off + u + 1);

    auto locate = [&](int it) {
        while (it >= u_last) { ++u; u_first = u_last; u_last = __ldg(prm.item_off + u + 1); }
        ItemRef r;
        const long long s0 = __ldg(prm.utt_off + u);
        r.n = (int)(__ldg(prm.utt_off + u + 1) - s0);
        r.f0 = __ldg(prm.frame_off + u);
        r.T = (int)(__ldg(prm.frame_off + u + 1) - r.f0);
        r.t0 = (it - u_first) * G::FPW;
        r.u = u;
        r.wav = prm.wav + s0;
        r.interior = item_is_interior<G>(r.n, r.t0, hop);
        return r;
    };
    auto prefetch = [&](const ItemRef& r) {                       // raw span + halo of an interior item -> stage[1 ..]
        const float* src = r.wav + ((long long)r.t0 * hop - G::PAD - 1);
        const int count = G::span(hop) + 2;
        for (int i = lane; i < count; i += 32) cp_async_f32(stage + G::LEAD - 1 + i, src + i);
        cp_async_commit();
    };

    ItemRef cur{};
    if (active) {
        cur = locate(item);
        if (cur.interior) prefetch(cur);
    }

    constexpr int n_streams = (MODE == kModeMfccPower) ? 2 : 1;
    for (; item < end; item = kDynamicItems ? item : item + kExtractWarps) {     // dynamic: advanced at the end of the body
        int item_next = end;
#pragma unroll 1
        for (int stream = 0; stream < n_streams; ++stream) {
            const int deriv = (MODE == kModeMfccPower) ? stream : prm.deriv;
            // One copy of the 25-point transform for both kinds of stream, or one straight-line block per kind?  With the
            // two instantiations the hot loop of the MFCC power kernel (both streams per item) held 27 KB of transform code
            // and missed the instruction cache on a fifth of its fetches; sharing the transform made it 5 % faster and the
            // n_fft 1600 kernel 3.8 % (smaller code), but costs the n_fft 800 dB kernel 1.8 % (one stream kind per launch:
            // nothing to share, and the join after the loads keeps them from overlapping the first butterflies).
            constexpr bool kSharedPass1 = !(R == 16 && MODE != kModeMfccPower);
            if constexpr (kSharedPass1) {
                if (cur.interior) {
                    if (stream == 0) { cp_async_wait_all(); __syncwarp(); }
                } else {
                    __syncwarp();
                    stage_item<G>(lane, cur.wav, cur.n, cur.t0, hop, deriv, stage);   // edge items: the stage already holds the stream
                    __syncwarp();
                }
                const bool diff = cur.interior && deriv != 0;
                if constexpr (FAST) {
                    WinRegs win;
                    win.load(taddr + TmemMap<R>::kWin);
                    pass1_shared<G>(lane, stage, hop, win, Y, diff);
                } else {
                    pass1_shared<G>(lane, stage, hop, WinShared{win2}, Y, diff);
                }
            } else {
                auto run_pass1 = [&](auto diff) {
                    if constexpr (FAST) {
                        WinRegs win;
                        win.load(taddr + TmemMap<R>::kWin);
                        pass1<G, decltype(diff)::value>(lane, stage, hop, win, Y);
                    } else {
                        pass1<G, decltype(diff)::value>(lane, stage, hop, WinShared{win2}, Y);
                    }
                };
                if (cur.interior) {
                    if (stream == 0) { cp_async_wait_all(); __syncwarp(); }
                    if (deriv) run_pass1(std::true_type{});
                    else run_pass1(std::false_type{});
                } else {
                    __syncwarp();
                    stage_item<G>(lane, cur.wav, cur.n, cur.t0, hop, deriv, stage);
                    __syncwarp();
                    run_pass1(std::false_type{});
                }
            }
            __syncwarp();                                        // stage is free, Y is complete

            ItemRef nxt = cur;
            if constexpr (kDynamicItems) {
                if (stream == n_streams - 1) {
                    item_next = grab();
                    if (item_next < end) {
                        nxt = locate(item_next);
                        if (nxt.interior) prefetch(nxt);         // overlaps pass 2, split and mel of this item
                    }
                }
            } else if (stream == n_streams - 1 && item + kExtractWarps < end) {
                nxt = locate(item + kExtractWarps);
                if (nxt.interior) prefetch(nxt);                 // overlaps pass 2, split and mel of this item
            }

            if constexpr (R <= 16) {
                // fused pass 2 + real split + power: rows j and 25-j stay in registers; the tile is overwritten by P only
                // after every lane has loaded its rows
                // Several rounds (n_fft 400: pairs 0-1, then pairs 2-3) run as a LOOP, each round storing its own power values:
                // round r's power tiles land on spectrum rows that rounds <= r have consumed (P of pairs 2r, 2r+1 lies below
                // the spectrum of pair 2r+2), so the rounds need no common barrier -- half the code (the unrolled form
                // stalled 0.95 cycles per issue on instruction fetch) and half the live registers
                constexpr int ROUNDS = G::PS_ROUNDS;
                static_assert(G::PP <= G::YP, "power tiles of pairs 0 .. 2r+1 must end before the spectrum tile of pair 2r+2 begins");
#pragma unroll 1
                for (int r = 0; r < ROUNDS; ++r) {
                    pk2 pu[R], pv[R];
                    int p, j;
                    if constexpr (FAST) {
                        // every lane runs the task (the twiddle fetch from tensor memory is warp-wide); lanes without one
                        // repeat row pair 12 of their frame pair (same addresses: broadcasts) and store nothing
                        G::ps_task(lane, r, p, j);
                        TwTmem tw{taddr + TmemMap<R>::kTw};
                        pass2_split<G>(p, j < 13 ? j : 12, Y, tw, pu, pv);
                    } else if (G::ps_task(lane, r, p, j)) {
                        TwShared tw{tws + j * G::TWS};
                        pass2_split<G>(p, j, Y, tw, pu, pv);
                    }
                    __syncwarp();
                    if (G::ps_task(lane, r, p, j)) pass2_split_store<G>(p, j, P, pu, pv);
                }
            } else {
#pragma unroll 1
                for (int task = lane; task < G::P2_TASKS; task += 32) pass2_row<G>(task, Y);
                __syncwarp();
                // real split + power: every Z of the item goes to registers, then the tile is overwritten by P
                pk2 a[13], b[13];
                bool on0 = false;
                TwTmem twt{taddr + TmemMap<R>::kTw};
                TwStrided tws_col{tws + lane % R, G::TWS};
#pragma unroll
                for (int k2 = 0; k2 <= 12; ++k2) {
                    bool on;
                    if constexpr (FAST) on = split_load<G>(lane, k2, Y, twt, a[k2], b[k2]);
                    else on = split_load<G>(lane, k2, Y, tws_col, a[k2], b[k2]);
                    if (k2 == 0) on0 = on;
                }
                __syncwarp();
                split_store_all<G>(lane, P, a, b, on0);
            }
            __syncwarp();

            // ---- mel bands (lane = band, all frame pairs of the item) + log + store --------------------------
            {
                const MelJob job{cur.f0, cur.T, cur.t0, cur.u, stream};
                if constexpr (FAST) mel_fast<G, MODE>(lane, P, taddr, prm, job);
                else mel_rounds<G, MODE>(lane, P, melp, n_mels, prm, job);
            }
            __syncwarp();                                        // P reads done before the next pass 1 overwrites Y
            if (stream == n_streams - 1) cur = nxt;
        }
        if constexpr (kDynamicItems) item = item_next;
    }
    if constexpr (FAST) {
        tmem::fence_before_sync();
        __syncthreads();
        if (warp == 0) tmem::dealloc(tmem_base, TmemMap<R>::kCols);
    }
}


// ---- host launchers ----------------------------------------------------------------------------------------
constexpr size_t kMaxSmem = kMaxDynSmem - 64;  // minus the static shared memory (tmem_base, cta_next)

template <int R>
static int extract_warps(int hop, int n_mel_entries) {
    using G = Geo<R>;
    return warps_that_fit(extract_const_bytes(R, n_mel_entries), G::stage_floats(hop) * 4 + G::Y_PK4 * 16,
                          ExtractWarps<R>::value, kMaxSmem);
}

template <int R>
static size_t extract_smem_bytes(int hop, int n_mel_entries) {
    using G = Geo<R>;
    const int w = extract_warps<R>(hop, n_mel_entries);
    if (w == 0) return kMaxSmem + 1;
    return (size_t)extract_const_bytes(R, n_mel_entries) + (size_t)w * (G::stage_floats(hop) * 4 + G::Y_PK4 * 16);
}

template <int R, int MODE>
static cudaError_t launch_one(const ExtractParams& prm, int grid, cudaStream_t stream) {
    const size_t smem = extract_smem_bytes<R>(prm.hop, prm.n_mel_entries);
    const int warps = extract_warps<R>(prm.hop, prm.n_mel_entries);
    auto kern = prm.mel_fast ? extract_kernel<R, MODE, true> : extract_kernel<R, MODE, false>;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kern<<<grid, warps * 32, smem, stream>>>(prm);
    return cudaGetLastError();
}

template <int R>
static cudaError_t launch_mode(const ExtractParams& prm, int mode, int grid, cudaStream_t stream) {
    switch (mode) {
        case kModeDbFrameMajor: return launch_one<R, kModeDbFrameMajor>(prm, grid, stream);
        case kModeDbBandMajor: return launch_one<R, kModeDbBandMajor>(prm, grid, stream);
        case kModeMfccPower: return launch_one<R, kModeMfccPower>(prm, grid, stream);
    }
    return cudaErrorInvalidValue;
}

cudaError_t launch_extract(const ExtractParams& prm, int n_fft, int mode, int grid, cudaStream_t stream) {
    switch (n_fft) {
        case 400: return launch_mode<8>(prm, mode, grid, stream);
        case 800: return launch_mode<16>(prm, mode, grid, stream);
        case 1600: return launch_mode<32>(prm, mode, grid, stream);
    }
    return cudaErrorInvalidValue;
}

int extract_frames_per_item(int n_fft) {
    switch (n_fft) {
        case 400: return Geo<8>::FPW;
        case 800: return Geo<16>::FPW;
        case 1600: return Geo<32>::FPW;
    }
    return 0;
}

size_t extract_smem_bytes_for(int n_fft, int hop, int n_mel_entries) {
    switch (n_fft) {
        case 400: return extract_smem_bytes<8>(hop, n_mel_entries);
        case 800: return extract_smem_bytes<16>(hop, n_mel_entries);
        case 1600: return extract_smem_bytes<32>(hop, n_mel_entries);
    }
    return 0;
}

}  // namespace sept
