// Per-lane phase functions of the log-mel backward: d(sum G * logmel) / d waveform (frame-major, deriv 0).
//
// Work unit: the forward's ITEM (FPW frames of one utterance, frame pairs packed in pk2), one warp per item.  For each
// item the frame pass (extract_bwd.cu)
//   1. recomputes the spectrum with the forward's own phase functions (stage_item, pass1, pass2_row) and splits it like
//      the forward (bwd_split: same operations, so 4|X|^2 and the recomputed mel power are the forward's bit for bit
//      and so is the clamp mask), keeping 2X in the spectrum tile;
//   2. recomputes the mel power with the forward's gather program (bwd_mel_sums) and forms
//      dM = G * 10 / (ln 10 * M), 0 where M < 1e-10 (bwd_dmel);
//   3. reads the gather program the other way: bin k of interval i gets dP = up dM[i] + dn dM[i-1] (bwd_dpower);
//   4. Z[k] = 2 dP[k] X[k] goes through the adjoint of the real split (bwd_unsplit) and the inverse prime-factor
//      transform, which is the forward's DFT-R and DFT-25 on conjugated data: IDFT(z) = conj(DFT(conj z)) -- pass2_row
//      over k1, then bwd_pass1 over k2, which also applies the window;
//   5. overlap-adds the item's frames into its span of (FPW-1)*hop + n_fft padded samples (bwd_ola) and writes that
//      span to a workspace row.
// The gather pass (bwd_gather) then sums, for every waveform sample, the span rows covering its padded position and
// the reflect-padded positions that mirror onto it, in a fixed order: no atomics, bit-deterministic.
//
// Like extract_core.cuh, everything here is __host__ __device__: tests/hostsim/logmel_bwd.cpp runs these functions
// lane by lane on the CPU against a float64 autograd oracle.
//
// Warp-private shared memory of the frame pass (floats):
//   stage  G::stage_floats(hop)         reflect-padded waveform span (forward staging)
//   Y      2 * G::Y_PK2                 spectrum tile of the forward; then 2X (Nyquist bin in row 0's pad), then
//                                       conj(H), then the windowed frame gradients F[FPW][n_fft] (time domain)
//   P      2 * PPW * PP                 4|X|^2 in the forward's power-tile layout; then dL/d(4|X|^2) in the same slots
//   U, D   2 * PPW * (n_mels + 1) each  per-interval rising / falling sums; U then holds dM per band
#pragma once
#include "extract_core.cuh"

namespace sept {

constexpr float kDbPerNeper = 4.34294481903251828f;      // 10 / ln 10: d(10 log10 M) / dM = kDbPerNeper / M

constexpr int kBwdWarps = 8;     // warps per CTA of the frame pass at most (shared memory decides: extract_bwd.cu)

#ifdef __CUDACC__                // kernel-side helpers of the frame passes (extract_bwd.cu, mfcc_bwd.cu)
// utterance u with off[u] <= x < off[u + 1] (off: item or sample offsets)
template <class Off>
__device__ __forceinline__ int bwd_find_utt(const Off* off, int n_utts, long long x) {
    int lo_ = 0, hi_ = n_utts - 1;
    while (lo_ < hi_) {
        const int mid = (lo_ + hi_) >> 1;
        if (__ldg(off + mid + 1) > x) hi_ = mid; else lo_ = mid + 1;
    }
    return lo_;
}

// bytes of the frame pass's shared constants (mel program, window, split twiddles) in front of the warp tiles
__host__ __device__ inline int bwd_const_bytes(int R, int n_mel_entries) {
    return (n_mel_entries * 16 + R * 25 * 8 + 13 * (R + 1) * 8 + 15) & ~15;
}
#endif

template <class G>
struct Bwd {
    static SEPT_HD int ums(int n_mels) { return n_mels + 1; }                 // pk2 per frame pair of U and D
    static SEPT_HD int row_floats(int hop) { return (G::span(hop) + 3) & ~3; } // workspace floats per item
    static SEPT_HD int ud_floats(int n_mels) { return (2 * G::PPW * ums(n_mels) + 3) & ~3; }
    static SEPT_HD int warp_floats(int hop, int n_mels) {
        return G::stage_floats(hop) + 2 * G::Y_PK2 + 2 * G::PPW * G::PP + 2 * ud_floats(n_mels);
    }
    static_assert(G::FPW * G::NFFT <= 2 * G::Y_PK2, "frame gradients must fit the spectrum tile");
    static_assert((2 * G::Y_PK2) % 4 == 0 && (2 * G::PPW * G::PP) % 4 == 0, "tiles stay 16-byte aligned");
};

// R <= 16: the forward keeps a copy of spectrum row 0 in row 25 and splits every bin of row 0 against that copy; copy
// the transformed row 0 there so that bwd_split can do the same
template <class G>
SEPT_HD void bwd_row0_copy(int lane, pk2* Y) {
    if constexpr (G::YROWS == 26)
    for (int i = lane; i < G::PPW * 2 * G::R; i += 32) {
        const int p = i / (2 * G::R), c = i % (2 * G::R);
        Y[p * G::YP + 25 * G::RS + c] = Y[p * G::YP + c];
    }
}

// lane (p, k1): for rows k2 = 0..12, the conjugate pairs Z[k], Z[NC-k] of the packed spectrum become 2X[k], 2X[NC-k]
// in place, and 4|X|^2 goes to the power tile.  The pairing, the twiddle and the operations are the forward's
// (split_pair; fused form for R <= 16, split_load / split_store_all for R = 32), so the power values are identical.
template <class G>
SEPT_HD void bwd_split(int lane, pk2* Y, const f2* tws, pk2* P) {
    constexpr int R = G::R, NC = G::NC, RS = G::RS;
    constexpr bool kRow0Copy = G::YROWS == 26;
    const int p = lane / R, k1 = lane % R, km = (R - k1) % R;
    pk2* y = Y + p * G::YP;
    pk2* pw = P + p * G::PP;
    int k = (Pfa<R>::cK1 * k1) % NC;
    for (int k2 = 0; k2 <= 12; ++k2) {
        if (k2 > 0 || kRow0Copy || k1 <= R / 2) {
            const int rb = k2 > 0 ? 25 - k2 : kRow0Copy ? 25 : 0;
            pk2* yk = y + k2 * RS + k1;
            pk2* ym = y + rb * RS + km;
            const pk4 zk{yk[0], yk[R]}, zm{ym[0], ym[R]};
            const f2 tw = tws[k2 * G::TWS + k1];
            const pk2 twr = splat(tw.x), twi = splat(tw.y);
            const pk2 er = zk.re + zm.re, ei = zk.im - zm.im;
            const pk2 o_r = zk.im + zm.im, o_i = zm.re - zk.re;
            const pk2 tr = fnma2(o_i, twi, o_r * twr), ti = fma2(o_i, twr, o_r * twi);
            const pk2 xr = er + tr, xi = ei + ti, yr = er - tr, yi = ei - ti;   // 2X[k]; conj of 2X[NC-k]
            if (k == 0) {                                                        // partner: the Nyquist bin
                pw[G::bin_pos(NC)] = fma2(yi, yi, yr * yr);
                y[2 * R] = yr;
                y[2 * R + 1] = neg(yi);
                for (int z = 0; z < G::ZSLOTS; ++z) pw[G::ZSLOT + z] = splat(0.f);
            } else if (k2 > 0 || !kRow0Copy) {                                   // own partner at NC/2: k wins below
                pw[G::bin_pos(NC - k)] = fma2(yi, yi, yr * yr);
                ym[0] = yr;
                ym[R] = neg(yi);
            }
            pw[G::bin_pos(k)] = fma2(xi, xi, xr * xr);
            yk[0] = xr;
            yk[R] = xi;
        }
        k += Pfa<R>::cK2;
        if (k >= NC) k -= NC;
    }
}

// mel power recomputed with the forward's gather program (mel_head / mel_round): U[p][i] = rising sum of interval i,
// D[p][i] = falling sum (band i-1); band m = U[m] + D[m+1], the forward's sum in the forward's order.  fast_dn: the
// compiled-in 128-band path of the forward takes the falling weight as 1/4 - rising (extract.cu: mel_round_regs).
template <class G>
SEPT_HD void bwd_mel_sums(int lane, const pk2* P, const mel_step* prog, int n_head, int n_mels, bool fast_dn, pk2* U,
                          pk2* D) {
    constexpr int PPW = G::PPW;
    const int ums = n_mels + 1, width = n_mels < 32 ? n_mels : 32;
    if (lane == 0) {
        pk2 h[PPW];
        mel_head<G>(P, prog, n_head, h);
        for (int p = 0; p < PPW; ++p) U[p * ums] = h[p];
    }
    const mel_step* e = prog + n_head + (lane < width ? lane : width - 1);
    const unsigned char* base = reinterpret_cast<const unsigned char*>(P);
    for (int m0 = 0; m0 < n_mels; m0 += 32) {
        const int n_steps = e->pad;
        if (m0 + lane < n_mels) {
            pk2 u[PPW], d[PPW];
            for (int p = 0; p < PPW; ++p) { u[p] = splat(0.f); d[p] = splat(0.f); }
            for (int s = 0; s < n_steps; ++s) {
                const mel_step st = e[s * width];
                const pk2 up = splat(st.up), dn = splat(fast_dn ? 0.25f - st.up : st.dn);
                for (int p = 0; p < PPW; ++p) {
                    const pk2 v = *reinterpret_cast<const pk2*>(base + st.off + p * (G::PP * 8));
                    u[p] = fma2(v, up, u[p]);
                    d[p] = fma2(v, dn, d[p]);
                }
            }
            const int i = 1 + m0 + lane;
            for (int p = 0; p < PPW; ++p) { U[p * ums + i] = u[p]; D[p * ums + i] = d[p]; }
        }
        e += n_steps * width;
    }
}

// dL/dM of one band value: the derivative of 10 log10(max(M, 1e-10)); torch.clamp passes the gradient where M >= min
SEPT_HD float bwd_dmel_one(float m, float g) { return m >= 1e-10f ? g * (kDbPerNeper / m) : 0.f; }

// lane = band: dM[p][m] = G * 10 / (ln 10 M) over U[p][m] (frames past the utterance: 0), dM[p][n_mels] = 0 (the last
// interval has no band above it); clears the power tile for bwd_dpower.  grad_u: the utterance's (T, n_mels) rows.
template <class G>
SEPT_HD void bwd_dmel(int lane, pk2* U, const pk2* D, const float* grad_u, int T, int t0, int n_mels, pk2* P) {
    const int ums = n_mels + 1;
    for (int m = lane; m < n_mels; m += 32)
        for (int p = 0; p < G::PPW; ++p) {
            const pk2 acc = U[p * ums + m] + D[p * ums + m + 1];
            const int ta = t0 + 2 * p;
            const float ga = ta < T ? grad_u[(long long)ta * n_mels + m] : 0.f;
            const float gb = ta + 1 < T ? grad_u[(long long)(ta + 1) * n_mels + m] : 0.f;
            U[p * ums + m] = pk(bwd_dmel_one(lo(acc), ga), bwd_dmel_one(hi(acc), gb));
        }
    if (lane == 0)
        for (int p = 0; p < G::PPW; ++p) U[p * ums + n_mels] = splat(0.f);
    for (int i = lane; i < G::PPW * G::PP; i += 32) P[i] = splat(0.f);
}

// the gather program read the other way: every bin of interval i (lane 1 + m0 + lane) gets
// dL/d(4|X|^2) = up dM[i] + dn dM[i-1] in its power-tile slot; interval 0 (head): up dM[0].  Each bin belongs to one
// interval, idle program slots point at the zero slots and are skipped; bins of no band (DC, Nyquist) stay 0.
template <class G>
SEPT_HD void bwd_dpower(int lane, const pk2* dM, const mel_step* prog, int n_head, int n_mels, pk2* P) {
    constexpr int PPW = G::PPW;
    const int ums = n_mels + 1, width = n_mels < 32 ? n_mels : 32;
    const int zoff = 8 * G::ZSLOT;
    if (lane == 0)
        for (int s = 0; s < n_head; ++s) {
            const mel_step st = prog[s];
            for (int p = 0; p < PPW; ++p) P[p * G::PP + st.off / 8] = splat(st.up) * dM[p * ums];
        }
    const mel_step* e = prog + n_head + (lane < width ? lane : width - 1);
    for (int m0 = 0; m0 < n_mels; m0 += 32) {
        const int n_steps = e->pad;
        if (m0 + lane < n_mels) {
            const int i = 1 + m0 + lane;
            for (int s = 0; s < n_steps; ++s) {
                const mel_step st = e[s * width];
                if (st.off >= zoff) continue;
                for (int p = 0; p < PPW; ++p)
                    P[p * G::PP + st.off / 8] = fma2(splat(st.dn), dM[p * ums + i - 1], splat(st.up) * dM[p * ums + i]);
            }
        }
        e += n_steps * width;
    }
}

// adjoint of the real split.  With dP = dL/d|X|^2 = 4 x (x: the power-tile gradient) and Z[k] = 2 dP[k] X[k], the frame gradient is
// g[n] = Re sum_{k=0..NC} Z[k] e^{+2 pi i k n / N}.  Its packed form h[m] = g[2m] + i g[2m+1] is the unnormalised
// inverse NC-point DFT of H[k] = E + iO, H[NC-k] = conj(E - iO), E = a + conj b, O = (a - conj b) e^{+2 pi i k / N},
// a = Z[k]/2, b = Z[NC-k]/2 (bins 0 and NC: the real part of Z, whole).  Lane (p, k1) takes the same conjugate pairs
// as bwd_split (row 0: k1 <= R/2) and writes conj(H) in place, ready for the forward transforms.
template <class G>
SEPT_HD void bwd_unsplit(int lane, pk2* Y, const pk2* P, const f2* tws) {
    constexpr int R = G::R, NC = G::NC, RS = G::RS;
    const int p = lane / R, k1 = lane % R, km = (R - k1) % R;
    pk2* y = Y + p * G::YP;
    const pk2* dt = P + p * G::PP;
    int k = (Pfa<R>::cK1 * k1) % NC;
    for (int k2 = 0; k2 <= 12; ++k2) {
        if (k2 > 0 || k1 <= R / 2) {
            pk2* yk = y + k2 * RS + k1;
            pk2* ym = y + ((25 - k2) % 25) * RS + km;
            const f2 tw = tws[k2 * G::TWS + k1];
            // a = Z[k] / 2 = dP[k] X[k] = (2 x[k]) (2X[k]) with the tile holding x = dP / 4 and 2X; bins 0 and NC: Re Z
            const pk2 sk = splat(2.f) * dt[G::bin_pos(k)], sm = splat(2.f) * dt[G::bin_pos(NC - k)];
            pk2 ar, ai, br, bi;
            if (k == 0) {
                ar = (sk + sk) * yk[0]; ai = splat(0.f);
                br = (sm + sm) * y[2 * R]; bi = splat(0.f);
            } else {
                ar = sk * yk[0]; ai = sk * yk[R];
                br = sm * ym[0]; bi = sm * ym[R];
            }
            const pk2 er = ar + br, ei = ai - bi, dr = ar - br, di = ai + bi;
            const pk2 twr = splat(tw.x), twi = splat(tw.y);       // W^k; e^{+2 pi i k / N} = conj(W^k)
            const pk2 o_r = fma2(di, twi, dr * twr), o_i = fnma2(dr, twi, di * twr);
            if (k != 0) { ym[0] = er + o_i; ym[R] = ei - o_r; }  // conj H[NC-k]; at NC/2 k's own value wins below
            yk[0] = er - o_i;
            yk[R] = neg(ei + o_r);                                // conj H[k]
        }
        k += Pfa<R>::cK2;
        if (k >= NC) k -= NC;
    }
}

// lane (p, n1): the DFT-25 over k2 of column n1 of the row-transformed tile gives conj(h) at m = (25 n1 + R n2) mod NC;
// h[m] = g[2m] + i g[2m+1], times the window.  Returns the lane's 25 windowed sample pairs (frame pair p).
template <class G>
SEPT_HD void bwd_pass1_load(int lane, const pk2* Y, const f2* win2, pk2 (&gr)[25], pk2 (&gi)[25]) {
    constexpr int R = G::R;
    const int p = lane / R, n1 = lane % R;
    const pk2* y = Y + p * G::YP + n1;
    pk2 re[25], im[25];
#pragma unroll
    for (int k2 = 0; k2 < 25; ++k2) { re[k2] = y[k2 * G::RS]; im[k2] = y[k2 * G::RS + R]; }
    Dft<25>::run(re, im);
#pragma unroll
    for (int n2 = 0; n2 < 25; ++n2) {
        const f2 w = win2[Pfa<R>::in_index(n1, n2)];
        gr[n2] = re[n2] * splat(w.x);
        gi[n2] = im[n2] * splat(-w.y);
    }
}

// ... and its store into the frame tile F[f][n] (overlays the spectrum tile: call after every lane has loaded)
template <class G>
SEPT_HD void bwd_pass1_store(int lane, float* F, const pk2 (&gr)[25], const pk2 (&gi)[25]) {
    constexpr int R = G::R, N = G::NFFT;
    const int p = lane / R, n1 = lane % R;
    float* fa = F + (2 * p) * N;
    float* fb = fa + N;
#pragma unroll
    for (int n2 = 0; n2 < 25; ++n2) {
        const int m = Pfa<R>::in_index(n1, n2);
        fa[2 * m] = lo(gr[n2]); fa[2 * m + 1] = lo(gi[n2]);
        fb[2 * m] = hi(gr[n2]); fb[2 * m + 1] = hi(gi[n2]);
    }
}

// overlap-add of the item's frames at span position j (padded index t0*hop + j), frames in order
template <class G>
SEPT_HD float bwd_ola(int j, const float* F, int hop) {
    float acc = 0.f;
    for (int f = 0; f < G::FPW; ++f) {
        const int o = j - f * hop;
        if (o >= 0 && o < G::NFFT) acc += F[f * G::NFFT + o];
    }
    return acc;
}

// gradient of sample s of an utterance of n samples: the span rows (ws_u: row 0 = the utterance's first item, `row`
// floats apart) at its own padded position s + pad and at the reflect-padded positions that mirror onto it, pad - s
// (1 <= s <= pad) and 2(n-1) - s + pad (s <= n-2); items in ascending order
template <class G>
SEPT_HD float bwd_gather(const float* ws_u, int row, int n_items, int n, int s, int hop) {
    const long long S = (long long)G::FPW * hop, span = G::span(hop);
    float acc = 0.f;
    auto add = [&](long long q) {
        long long j = q < span ? 0 : (q - span) / S + 1;
        long long j_end = q / S;
        if (j_end > n_items - 1) j_end = n_items - 1;
        for (; j <= j_end; ++j) acc += ws_u[j * row + (q - j * S)];
    };
    add((long long)s + G::PAD);
    if (s >= 1 && s <= G::PAD) add((long long)G::PAD - s);
    if (s <= n - 2) add(2LL * (n - 1) - s + G::PAD);
    return acc;
}

}  // namespace sept
