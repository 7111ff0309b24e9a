// Host build of the training-window multiplicity shared by the statistics kernels and their backward
// (csrc/norm_weight.cuh), compiled with -D__device__= -D__forceinline__=inline.
//   norm_weight weights <win> <shift> <T_max> <whole> <out.bin>
//       for T = 1 .. T_max and t = 0 .. T-1: frame_weight, then (a second array) frame_weight_fast with the inv_shift
//       and n_win the kernels pass it; int32, T-major
//   norm_weight div <d> ...
//       div_floor_small(a, d, 1.0f / d) against a / d for every 0 <= a < 2^22; prints "mismatches <n>" and the first few
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "norm_weight.cuh"

static int weights(int win, int shift, int T_max, bool whole, const char* path) {
    std::vector<int32_t> slow, fast;
    const float inv_shift = 1.0f / (float)shift;
    for (int T = 1; T <= T_max; ++T) {
        const int n_win = T >= win ? (T - win) / shift + 1 : 0;       // as utt_partial128_kernel / stats_bwd_* compute it
        for (int t = 0; t < T; ++t) {
            slow.push_back(sept::frame_weight(t, T, win, shift, whole));
            fast.push_back(sept::frame_weight_fast(t, T, win, shift, inv_shift, n_win, whole));
        }
    }
    FILE* f = std::fopen(path, "wb");
    if (!f) return 2;
    std::fwrite(slow.data(), 4, slow.size(), f);
    std::fwrite(fast.data(), 4, fast.size(), f);
    std::fclose(f);
    return 0;
}

static int div_check(int argc, char** argv) {
    long long bad = 0;
    for (int i = 2; i < argc; ++i) {
        const int d = std::atoi(argv[i]);
        const float inv = 1.0f / (float)d;
        for (int a = 0; a < (1 << 22); ++a) {
            const int q = sept::div_floor_small(a, d, inv);
            if (q != a / d) {
                if (bad < 5) std::printf("a %d d %d got %d want %d\n", a, d, q, a / d);
                ++bad;
            }
        }
    }
    std::printf("mismatches %lld\n", bad);
    return 0;
}

int main(int argc, char** argv) {
    if (argc >= 3 && !std::strcmp(argv[1], "div")) return div_check(argc, argv);
    if (argc == 7 && !std::strcmp(argv[1], "weights"))
        return weights(std::atoi(argv[2]), std::atoi(argv[3]), std::atoi(argv[4]), std::atoi(argv[5]) != 0, argv[6]);
    return 1;
}
