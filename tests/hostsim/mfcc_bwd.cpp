// Host emulation of the MFCC backward (TEST CODE, not a fallback) for ONE utterance: the mel power of both streams with
// the frame pass's own recompute (extract_bwd.cuh), the head functions of csrc/mfcc_bwd.cuh per (frame, band), the
// route (floor totals, argmax share), the frame pass of the waveform and of the np.gradient stream (deriv staging) lane
// by lane as in extract_bwd.cu / mfcc_bwd.cu, then the gather with the np.gradient adjoint sample by sample.
//   mfcc_bwd grad <wav.f32> <gbar.f32 (120, T)> <dwav.f32>
//   mfcc_bwd adjoint <x.f32> <v.f32> <out.f32>     out = [np.gradient(x) as staged (n), its adjoint applied to v (n)]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "mfcc_bwd.cuh"
#include "tables.h"

using namespace sept;
using G = Geo<8>;
using B = Bwd<G>;

static constexpr int kHop = 200, kMels = 128;

struct Frames {
    std::vector<float> win, tws;
    MelProgram prog;
    const mel_step* mprog;
    bool fast_dn;
    std::vector<float> stage;
    std::vector<pk4> Ybuf, Pbuf;
    std::vector<pk2> U, D;
    pk2 *Y, *P;
    Frames() {
        win = make_hann_periodic(400);
        tws = make_split_twiddles(400);
        make_mel_program(400, kMels, 16000, prog);
        mprog = reinterpret_cast<const mel_step*>(prog.entries.data());
        fast_dn = prog.round_steps.size() == 4 && prog.n_head == FastMel<8>::head && prog.round_steps[0] == FastMel<8>::s0 &&
                  prog.round_steps[1] == FastMel<8>::s1 && prog.round_steps[2] == FastMel<8>::s2 &&
                  prog.round_steps[3] == FastMel<8>::s3;
        stage.assign(G::stage_floats(kHop), 0.f);
        Ybuf.resize(G::Y_PK4 + 1);
        Pbuf.resize((G::PPW * G::PP) / 2 + 1);
        U.resize((size_t)G::PPW * B::ums(kMels));
        D.resize((size_t)G::PPW * B::ums(kMels));
        Y = reinterpret_cast<pk2*>(Ybuf.data());
        P = reinterpret_cast<pk2*>(Pbuf.data());
    }
    const f2* win2() const { return reinterpret_cast<const f2*>(win.data()); }
    const f2* tw2() const { return reinterpret_cast<const f2*>(tws.data()); }
    // spectrum, split and mel sums of one item (the first half of the frame pass)
    void front(const std::vector<float>& wav, int t0, int deriv) {
        const int n = (int)wav.size();
        for (int lane = 0; lane < 32; ++lane) stage_item<G>(lane, wav.data(), n, t0, kHop, deriv, stage.data());
        for (int lane = 0; lane < 32; ++lane) pass1<G, false>(lane, stage.data(), kHop, WinShared{win2()}, Y);
        for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_row0_copy<G>(lane, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_split<G>(lane, Y, tw2(), P);
        for (int lane = 0; lane < 32; ++lane) bwd_mel_sums<G>(lane, P, mprog, prog.n_head, kMels, fast_dn, U.data(), D.data());
    }
    // mel power (T, 128) of the stream
    std::vector<float> power(const std::vector<float>& wav, int T, int deriv) {
        std::vector<float> M((size_t)T * kMels, 0.f);
        const int ums = kMels + 1;
        for (int t0 = 0; t0 < T; t0 += G::FPW) {
            front(wav, t0, deriv);
            for (int p = 0; p < G::PPW; ++p)
                for (int m = 0; m < kMels; ++m) {
                    const pk2 acc = U[p * ums + m] + D[p * ums + m + 1];
                    if (t0 + 2 * p < T) M[(size_t)(t0 + 2 * p) * kMels + m] = lo(acc);
                    if (t0 + 2 * p + 1 < T) M[(size_t)(t0 + 2 * p + 1) * kMels + m] = hi(acc);
                }
        }
        return M;
    }
    // the whole frame pass: span rows of every item for dB gradient grad (T, 128)
    std::vector<float> rows(const std::vector<float>& wav, int T, int deriv, const std::vector<float>& grad) {
        const int n_items = (T + G::FPW - 1) / G::FPW, row = B::row_floats(kHop);
        std::vector<float> ws((size_t)n_items * row, 0.f);
        static pk2 gr[32][25], gi[32][25];
        for (int it = 0; it < n_items; ++it) {
            const int t0 = it * G::FPW;
            front(wav, t0, deriv);
            for (int lane = 0; lane < 32; ++lane) bwd_dmel<G>(lane, U.data(), D.data(), grad.data(), T, t0, kMels, P);
            for (int lane = 0; lane < 32; ++lane) bwd_dpower<G>(lane, U.data(), mprog, prog.n_head, kMels, P);
            for (int lane = 0; lane < 32; ++lane) bwd_unsplit<G>(lane, Y, P, tw2());
            for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
            for (int lane = 0; lane < 32; ++lane) bwd_pass1_load<G>(lane, Y, win2(), gr[lane], gi[lane]);
            for (int lane = 0; lane < 32; ++lane) bwd_pass1_store<G>(lane, reinterpret_cast<float*>(Y), gr[lane], gi[lane]);
            for (int j = 0; j < G::span(kHop); ++j) ws[(size_t)it * row + j] = bwd_ola<G>(j, reinterpret_cast<const float*>(Y), kHop);
        }
        return ws;
    }
};

static unsigned bits(float x) { unsigned u; std::memcpy(&u, &x, 4); return u; }

static std::vector<float> mfcc_grad(const std::vector<float>& wav, const std::vector<float>& gbar) {
    const int n = (int)wav.size(), T = 1 + n / kHop, n_items = (T + G::FPW - 1) / G::FPW;
    Frames fr;
    const std::vector<float> M0 = fr.power(wav, T, 0), M1 = fr.power(wav, T, 1);
    float max0 = 0.f, max1 = 0.f;                           // the forward's atomicMax over non-negative bits
    for (size_t i = 0; i < M0.size(); ++i) { max0 = M0[i] > max0 ? M0[i] : max0; max1 = M1[i] > max1 ? M1[i] : max1; }
    const MfccFloors fl = mfcc_floors(max0, max1);
    const std::vector<float> dct = make_dct_ortho(kMfccCoefs, kMels);
    std::vector<float> G0((size_t)T * kMels), G1((size_t)T * kMels);
    float R[3] = {0.f, 0.f, 0.f};
    int c0 = 0, c1 = 0;
    for (int f = 0; f < T; ++f) {
        float part[3] = {0.f, 0.f, 0.f};
        for (int b = 0; b < kMels; ++b) {
            const size_t i = (size_t)f * kMels + b;
            const MfccHead h = mfcc_head_one([&](int r) { return gbar[(size_t)r * T + f]; }, dct.data() + b * kMfccCoefs,
                                             M0[i], M1[i], fl);
            G0[i] = h.g0;
            G1[i] = h.g1;
            for (int s = 0; s < 3; ++s) part[s] += h.r[s];
            c0 += bits(M0[i]) == bits(max0);
            c1 += bits(M1[i]) == bits(max1);
        }
        for (int s = 0; s < 3; ++s) R[s] += part[s];
    }
    const float s0 = R[0] / (float)c0, s1 = R[1] / (float)c1, s2 = R[2] / (float)c1;
    for (size_t i = 0; i < G0.size(); ++i) {
        if (bits(M0[i]) == bits(max0)) mfcc_add_share0(G0[i], s0);
        if (bits(M1[i]) == bits(max1)) mfcc_add_share1(G1[i], s1, s2, max1);
    }
    const std::vector<float> ws0 = fr.rows(wav, T, 0, G0), ws1 = fr.rows(wav, T, 1, G1);
    std::vector<float> dwav(n);
    for (int s = 0; s < n; ++s) dwav[s] = mfcc_bwd_gather(ws0.data(), ws1.data(), B::row_floats(kHop), n_items, n, s);
    return dwav;
}

static bool read_f32(const char* path, std::vector<float>& v) {
    FILE* f = std::fopen(path, "rb");
    if (!f) return false;
    std::fseek(f, 0, SEEK_END);
    const long bytes = std::ftell(f);
    std::fseek(f, 0, SEEK_SET);
    v.resize(bytes / 4);
    const bool ok = std::fread(v.data(), 4, v.size(), f) == v.size();
    std::fclose(f);
    return ok;
}

int main(int argc, char** argv) {
    if (argc != 5) return 1;
    std::vector<float> a, b, out;
    if (!read_f32(argv[2], a) || !read_f32(argv[3], b)) return 2;
    const int n = (int)a.size();
    if (!std::strcmp(argv[1], "grad")) {
        if ((long long)b.size() != (long long)kMfccRows * (1 + n / kHop)) return 4;
        out = mfcc_grad(a, b);
    } else if (!std::strcmp(argv[1], "adjoint")) {
        if ((int)b.size() != n) return 4;
        out.resize(2 * (size_t)n);
        for (int s = 0; s < n; ++s) out[s] = staged_sample(a.data(), n, s, 1);
        for (int s = 0; s < n; ++s) out[n + s] = np_gradient_adjoint([&](int j) { return b[j]; }, n, s);
    } else {
        return 3;
    }
    FILE* f = std::fopen(argv[4], "wb");
    if (!f) return 2;
    std::fwrite(out.data(), sizeof(float), out.size(), f);
    std::fclose(f);
    return 0;
}
