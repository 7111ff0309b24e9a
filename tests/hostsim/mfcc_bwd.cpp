// Host emulation of the MFCC backward (TEST CODE, not a fallback) for ONE utterance: the mel power of both streams with
// the frame pass's own recompute (extract_bwd.cuh), the head functions of csrc/mfcc_bwd.cuh per (frame, band), the
// route (floor totals, argmax share), the frame pass of the waveform and of the np.gradient stream (deriv staging) lane
// by lane (bwd_frame_pass.h), then the gather with the np.gradient adjoint sample by sample.
//   mfcc_bwd grad <wav.f32> <gbar.f32 (120, T)> <dwav.f32>
//   mfcc_bwd adjoint <x.f32> <v.f32> <out.f32>     out = [np.gradient(x) as staged (n), its adjoint applied to v (n)]
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "bwd_frame_pass.h"
#include "mfcc_bwd.cuh"

using namespace sept;
using G = Geo<8>;
using B = Bwd<G>;

static constexpr int kHop = 200, kMels = 128;

static unsigned bits(float x) { unsigned u; std::memcpy(&u, &x, 4); return u; }

static std::vector<float> mfcc_grad(const std::vector<float>& wav, const std::vector<float>& gbar) {
    const int n = (int)wav.size(), T = 1 + n / kHop, n_items = (T + G::FPW - 1) / G::FPW;
    BwdFramePass<8> fr(kHop, kMels);
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
