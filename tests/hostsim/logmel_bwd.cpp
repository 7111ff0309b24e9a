// Host emulation of the log-mel backward (TEST CODE, not a fallback) for ONE utterance: the frame pass lane by lane
// (bwd_frame_pass.h), then the gather pass sample by sample.
//   logmel_bwd <n_fft> <hop> <n_mels> <wav.f32> <grad.f32 (T, n_mels)> <dwav.f32>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "bwd_frame_pass.h"

using namespace sept;

template <int R>
int run(int hop, int n_mels, const std::vector<float>& wav, const std::vector<float>& grad, const char* out_path) {
    using G = Geo<R>;
    const int n = (int)wav.size(), T = 1 + n / hop, n_items = (T + G::FPW - 1) / G::FPW;
    if ((long long)grad.size() != (long long)T * n_mels) return 4;
    const std::vector<float> ws = BwdFramePass<R>(hop, n_mels).rows(wav, T, 0, grad);
    const int row = Bwd<G>::row_floats(hop);
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
