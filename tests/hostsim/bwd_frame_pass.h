// Host emulation of the backward's frame pass (TEST CODE, not a fallback), shared by logmel_bwd.cpp and mfcc_bwd.cpp:
// the per-lane phase functions of csrc/extract_bwd.cuh (with the forward's own from extract_core.cuh) in loops over lane
// ids, in the order and with the warp barriers of logmel_bwd_frames_kernel (extract_bwd.cu), for ONE utterance.
#pragma once
#include <vector>

#include "extract_bwd.cuh"
#include "tables.h"

namespace sept {

template <int R>
struct BwdFramePass {
    using G = Geo<R>;
    using B = Bwd<G>;
    const int hop, n_mels;
    std::vector<float> win, tws;
    MelProgram prog;
    const mel_step* mprog;
    bool fast_dn;                // the forward runs its compiled-in 128-band path (ExtractParams::mel_fast)
    std::vector<float> stage;
    std::vector<pk4> Ybuf, Pbuf;
    std::vector<pk2> U, D;
    pk2 *Y, *P;

    BwdFramePass(int hop, int n_mels)
        : hop(hop), n_mels(n_mels), win(make_hann_periodic(G::NFFT)), tws(make_split_twiddles(G::NFFT)),
          stage(G::stage_floats(hop), 0.f), Ybuf(G::Y_PK4 + 1), Pbuf((G::PPW * G::PP) / 2 + 1),
          U((size_t)G::PPW * B::ums(n_mels)), D((size_t)G::PPW * B::ums(n_mels)) {
        make_mel_program(G::NFFT, n_mels, 16000, prog);
        mprog = reinterpret_cast<const mel_step*>(prog.entries.data());
        fast_dn = extract_mel_fast_ok(G::NFFT, n_mels, prog.n_head, prog.round_steps.data(), (int)prog.round_steps.size());
        Y = reinterpret_cast<pk2*>(Ybuf.data());
        P = reinterpret_cast<pk2*>(Pbuf.data());
    }
    const f2* win2() const { return reinterpret_cast<const f2*>(win.data()); }
    const f2* tw2() const { return reinterpret_cast<const f2*>(tws.data()); }

    // spectrum, split and mel sums of the item at frame t0 (the first half of the frame pass)
    void front(const std::vector<float>& wav, int t0, int deriv) {
        const int n = (int)wav.size();
        for (int lane = 0; lane < 32; ++lane) stage_item<G>(lane, wav.data(), n, t0, hop, deriv, stage.data());
        for (int lane = 0; lane < 32; ++lane) pass1<G, false>(lane, stage.data(), hop, WinShared{win2()}, Y);
        for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_row0_copy<G>(lane, Y);
        for (int lane = 0; lane < 32; ++lane) bwd_split<G>(lane, Y, tw2(), P);
        for (int lane = 0; lane < 32; ++lane) bwd_mel_sums<G>(lane, P, mprog, prog.n_head, n_mels, fast_dn, U.data(), D.data());
    }

    // mel power (T, n_mels) of the stream
    std::vector<float> power(const std::vector<float>& wav, int T, int deriv) {
        std::vector<float> M((size_t)T * n_mels, 0.f);
        const int ums = n_mels + 1;
        for (int t0 = 0; t0 < T; t0 += G::FPW) {
            front(wav, t0, deriv);
            for (int p = 0; p < G::PPW; ++p)
                for (int m = 0; m < n_mels; ++m) {
                    const pk2 acc = U[p * ums + m] + D[p * ums + m + 1];
                    if (t0 + 2 * p < T) M[(size_t)(t0 + 2 * p) * n_mels + m] = lo(acc);
                    if (t0 + 2 * p + 1 < T) M[(size_t)(t0 + 2 * p + 1) * n_mels + m] = hi(acc);
                }
        }
        return M;
    }

    // the whole frame pass: span rows of every item for the dB gradient grad (T, n_mels)
    std::vector<float> rows(const std::vector<float>& wav, int T, int deriv, const std::vector<float>& grad) {
        const int n_items = (T + G::FPW - 1) / G::FPW, row = B::row_floats(hop);
        std::vector<float> ws((size_t)n_items * row, 0.f);
        static pk2 gr[32][25], gi[32][25];
        for (int it = 0; it < n_items; ++it) {
            const int t0 = it * G::FPW;
            front(wav, t0, deriv);
            for (int lane = 0; lane < 32; ++lane) bwd_dmel<G>(lane, U.data(), D.data(), grad.data(), T, t0, n_mels, P);
            for (int lane = 0; lane < 32; ++lane) bwd_dpower<G>(lane, U.data(), mprog, prog.n_head, n_mels, P);
            for (int lane = 0; lane < 32; ++lane) bwd_unsplit<G>(lane, Y, P, tw2());
            for (int task = 0; task < G::P2_TASKS; ++task) pass2_row<G>(task, Y);
            for (int lane = 0; lane < 32; ++lane) bwd_pass1_load<G>(lane, Y, win2(), gr[lane], gi[lane]);
            for (int lane = 0; lane < 32; ++lane) bwd_pass1_store<G>(lane, reinterpret_cast<float*>(Y), gr[lane], gi[lane]);
            for (int j = 0; j < G::span(hop); ++j) ws[(size_t)it * row + j] = bwd_ola<G>(j, reinterpret_cast<const float*>(Y), hop);
        }
        return ws;
    }
};

}  // namespace sept
