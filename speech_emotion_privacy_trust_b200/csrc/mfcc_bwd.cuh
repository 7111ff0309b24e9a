// Per-element functions of the MFCC backward: d(sum Gbar * mfcc) / d waveform for the (120, T) blocks of sept_mfcc_f32.
//
// For stream s (0: x, 1: g = np.gradient(x), 2: g / 2) the forward computes, per utterance,
//   M_s = mel power, L_s = 10 log10(max(M_s, 1e-10)), m_s = max L_s, F_s = max(L_s, m_s - 80), out[40 s + c] = F_s @ D.
// Its gradient, what torch autograd gives for that composition:
//   1. Fbar_s[f][b] = sum_c D[b][c] Gbar[40 s + c][f]                                  (DCT adjoint, mfcc_head_one)
//   2. torch.maximum: Fbar passes to Lbar_s where L_s > m_s - 80, goes to the floor where L_s < m_s - 80, half each at a
//      tie (mfcc_floor_route).  The floor's total R_s reaches m_s and through amax the argmax positions of L_s, split
//      evenly among ties (added by the route pass, mfcc_bwd.cu).
//   3. the clamp and the power: the log-mel frame pass (extract_bwd.cuh) on dB gradient Lbar.
//   4. stream 2 folds into stream 1: M_2 = M_1 / 4 exactly, and d dB(P(a g)) / dg = d dB(P(g)) / dg, so
//      G_1 = Lbar_1 + Lbar_2 [M_1 / 4 >= 1e-10] runs through stream 1's frame pass; its argmax set is stream 1's.
//   5. dx = Bwd(x, G_0) + grad^T Bwd(g, G_1), grad^T the adjoint of np.gradient (np_gradient_adjoint).
//
// The masks are taken on the forward's own fp32 values: the recomputed power is the forward's bit for bit, dB is
// mfcc_dct.cu's (lg2.approx.ftz; log2f in the host emulation), and the argmax set is the positions whose power
// bit-equals the utterance maximum the forward's power kernel found.
//
// __host__ __device__ like extract_core.cuh: tests/hostsim/mfcc_bwd.cpp runs them on the CPU against a float64 oracle.
#pragma once
#include <cmath>
#include <cstdint>

#include "extract_bwd.cuh"

namespace sept {

constexpr int kMfccBands = 128, kMfccCoefs = 40, kMfccRows = 3 * kMfccCoefs;
constexpr float kMfccTopDb = 80.0f;
constexpr float kMfccDbQuarter = 6.02059991327962390f;   // 10 log10(4): stream 2's dB is stream 1's minus this
constexpr float kMfccDbPerLog2 = 3.01029995663981195f;   // 10 log10(2)
constexpr float kMfccDbMin = -100.0f;                    // 10 log10(amin)

// clamped dB of one mel power, as mfcc_dct.cu's db_clamped(p, -100)
SEPT_HD float mfcc_db(float p) {
    float l;
#ifdef __CUDA_ARCH__
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(p));
#else
    l = std::log2(p);
#endif
    return fmaxf(kMfccDbPerLog2 * l, kMfccDbMin);
}

// m_s - 80 of the three streams from the utterance's maximum mel power of streams 0 and 1
struct MfccFloors { float f0, f1, f2; };
SEPT_HD MfccFloors mfcc_floors(float max0, float max1) {
    const float m0 = mfcc_db(max0), m1 = mfcc_db(max1), m2 = fmaxf(m1 - kMfccDbQuarter, kMfccDbMin);
    return {m0 - kMfccTopDb, m1 - kMfccTopDb, m2 - kMfccTopDb};
}

// torch.maximum(L, floor) backward: pass where L > floor, to the floor where L < floor, half each at a tie
SEPT_HD void mfcc_floor_route(float L, float floor_db, float g, float& pass, float& floored) {
    if (L > floor_db) { pass = g; floored = 0.f; }
    else if (L < floor_db) { pass = 0.f; floored = g; }
    else { pass = 0.5f * g; floored = 0.5f * g; }
}

// stream 2's clamp mask in stream 1's terms: M_2 = M_1 / 4 >= 1e-10 (the scaling by 1/4 is exact)
SEPT_HD bool mfcc_quarter_live(float m1) { return m1 * 0.25f >= 1e-10f; }

// one (frame, band): the DCT adjoint of the three streams, the floor routing, the stream fold.
//   gbar(r)  upstream gradient of row r (0..119) of the frame;  d: D[b][0..39];  p0, p1: mel power of streams 0, 1
// g0, g1: the dB gradients of the frame passes before the argmax share; r[s]: what stream s sends to its floor.
struct MfccHead { float g0, g1, r[3]; };
template <class GBar>
SEPT_HD MfccHead mfcc_head_one(GBar gbar, const float* d, float p0, float p1, const MfccFloors& fl) {
    float fb[3] = {0.f, 0.f, 0.f};
    for (int s = 0; s < 3; ++s)
        for (int c = 0; c < kMfccCoefs; ++c) fb[s] = fmaf(d[c], gbar(kMfccCoefs * s + c), fb[s]);
    const float L0 = mfcc_db(p0), L1 = mfcc_db(p1), L2 = fmaxf(L1 - kMfccDbQuarter, kMfccDbMin);
    MfccHead h;
    float pass0, pass1, pass2;
    mfcc_floor_route(L0, fl.f0, fb[0], pass0, h.r[0]);
    mfcc_floor_route(L1, fl.f1, fb[1], pass1, h.r[1]);
    mfcc_floor_route(L2, fl.f2, fb[2], pass2, h.r[2]);
    h.g0 = pass0;
    h.g1 = mfcc_quarter_live(p1) ? pass1 + pass2 : pass1;
    return h;
}

// the argmax share, added to the head's values at the positions whose power bit-equals the utterance maximum:
// share[s] = R_s / (number of such positions of stream s; stream 2 counts stream 1's)
SEPT_HD void mfcc_add_share0(float& g0, float share0) { g0 += share0; }
SEPT_HD void mfcc_add_share1(float& g1, float share1, float share2, float max1) {
    g1 += mfcc_quarter_live(max1) ? share1 + share2 : share1;
}

// adjoint of np.gradient (edge_order 1, n >= 4) at sample s: v(j) = d/d g[j]
//   g[0] = x1 - x0,  g[j] = (x[j+1] - x[j-1]) / 2,  g[n-1] = x[n-1] - x[n-2]
template <class V>
SEPT_HD float np_gradient_adjoint(V v, int n, int s) {
    if (s == 0) return -v(0) - 0.5f * v(1);
    if (s == 1) return v(0) - 0.5f * v(2);
    if (s == n - 2) return 0.5f * v(n - 3) - v(n - 1);
    if (s == n - 1) return 0.5f * v(n - 2) + v(n - 1);
    return 0.5f * v(s - 1) - 0.5f * v(s + 1);
}

// gradient of sample s of an utterance: stream 0's rows at s, then grad^T of stream 1's per-sample sums, which the
// gather recomputes at s - 1 and s + 1 (edges: the formulas above) from the same span rows
SEPT_HD float mfcc_bwd_gather(const float* ws0_u, const float* ws1_u, int row, int n_items, int n, int s) {
    using G = Geo<8>;
    const float a = bwd_gather<G>(ws0_u, row, n_items, n, s, 200);
    auto v = [&](int j) { return bwd_gather<G>(ws1_u, row, n_items, n, j, 200); };
    return a + np_gradient_adjoint(v, n, s);
}

}  // namespace sept
