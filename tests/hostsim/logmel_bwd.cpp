// Host emulation of the log-mel backward (TEST CODE, not a fallback): runs the per-lane phase functions of the frame
// pass (csrc/extract_bwd.cuh, with the forward's own from extract_core.cuh) in loops over lane ids, in the order and with
// the warp barriers of extract_bwd.cu, then the gather pass sample by sample, for ONE utterance.
//   logmel_bwd <n_fft> <hop> <n_mels> <wav.f32> <grad.f32 (T, n_mels)> <dwav.f32>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "extract_bwd.cuh"
#include "tables.h"

using namespace sept;

template <int R>
int run(int hop, int n_mels, const std::vector<float>& wav, const std::vector<float>& grad, const char* out_path) {
    using G = Geo<R>;
    using B = Bwd<G>;
    const int n = (int)wav.size(), n_fft = G::NFFT;
    const int T = 1 + n / hop, n_items = (T + G::FPW - 1) / G::FPW;
    if ((long long)grad.size() != (long long)T * n_mels) return 4;
    std::vector<float> win = make_hann_periodic(n_fft), tws = make_split_twiddles(n_fft);
    MelProgram prog;
    make_mel_program(n_fft, n_mels, 16000, prog);
    const mel_step* mprog = reinterpret_cast<const mel_step*>(prog.entries.data());
    const bool fast_dn = n_mels == 128 && prog.round_steps.size() == 4 && prog.n_head == FastMel<R>::head &&
                         prog.round_steps[0] == FastMel<R>::s0 && prog.round_steps[1] == FastMel<R>::s1 &&
                         prog.round_steps[2] == FastMel<R>::s2 && prog.round_steps[3] == FastMel<R>::s3;
    const f2* win2 = reinterpret_cast<const f2*>(win.data());
    const f2* tw2 = reinterpret_cast<const f2*>(tws.data());
    std::vector<float> stage(G::stage_floats(hop), 0.f);
    std::vector<pk4> Ybuf(G::Y_PK4 + 1), Pbuf((G::PPW * G::PP) / 2 + 1);
    std::vector<pk2> U((size_t)G::PPW * B::ums(n_mels)), D((size_t)G::PPW * B::ums(n_mels));
    pk2* Y = reinterpret_cast<pk2*>(Ybuf.data());
    pk2* P = reinterpret_cast<pk2*>(Pbuf.data());
    const int row = B::row_floats(hop);
    std::vector<float> ws((size_t)n_items * row, 0.f);
    static pk2 gr[32][25], gi[32][25];
    for (int it = 0; it < n_items; ++it) {
        const int t0 = it * G::FPW;
        for (int lane = 0; lane < 32; ++lane) stage_item<G>(lane, wav.data(), n, t0, hop, 0, stage.data());
        for (int lane = 0; lane < 32; ++lane) pass1<G, false>(lane, stage.data(), hop, WinShared{win2}, Y);
        for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_row0_copy<G>(lane, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_split<G>(lane, Y, tw2, P);
        for (int lane = 0; lane < 32; ++lane) bwd_mel_sums<G>(lane, P, mprog, prog.n_head, n_mels, fast_dn, U.data(), D.data());
        for (int lane = 0; lane < 32; ++lane) bwd_dmel<G>(lane, U.data(), D.data(), grad.data(), T, t0, n_mels, P);
        for (int lane = 0; lane < 32; ++lane) bwd_dpower<G>(lane, U.data(), mprog, prog.n_head, n_mels, P);
        for (int lane = 0; lane < 32; ++lane) bwd_unsplit<G>(lane, Y, P, tw2);
        for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_pass1_load<G>(lane, Y, win2, gr[lane], gi[lane]);
        for (int lane = 0; lane < 32; ++lane) bwd_pass1_store<G>(lane, reinterpret_cast<float*>(Y), gr[lane], gi[lane]);
        for (int j = 0; j < G::span(hop); ++j) ws[(size_t)it * row + j] = bwd_ola<G>(j, reinterpret_cast<const float*>(Y), hop);
    }
    std::vector<float> dwav(n);
    for (int s = 0; s < n; ++s) dwav[s] = bwd_gather<G>(ws.data(), row, n_items, n, s, hop);
    FILE* f = std::fopen(out_path, "wb");
    if (!f) return 2;
    std::fwrite(dwav.data(), sizeof(float), dwav.size(), f);
    std::fclose(f);
    return 0;
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
    if (argc != 7) return 1;
    const int n_fft = std::atoi(argv[1]), hop = std::atoi(argv[2]), n_mels = std::atoi(argv[3]);
    std::vector<float> wav, grad;
    if (!read_f32(argv[4], wav) || !read_f32(argv[5], grad)) return 2;
    switch (n_fft) {
        case 400: return run<8>(hop, n_mels, wav, grad, argv[6]);
        case 800: return run<16>(hop, n_mels, wav, grad, argv[6]);
        case 1600: return run<32>(hop, n_mels, wav, grad, argv[6]);
    }
    return 3;
}
