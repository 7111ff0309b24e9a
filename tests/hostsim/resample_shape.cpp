// Launch configuration of the sinc resampler for a rate pair (TEST CODE): computed with the library's own functions
// (tables.h: make_resample_rows, make_resample_tiles; resample_shape.h: resample_shape), so a test can name the kernel
// path a rate pair takes and notice when a tiling change moves it.
//   resample_shape <orig_freq> <new_freq>      prints "orig <o> up <u> width <w> taps <t> n_groups <g> tg <tg>
//                                              group_span <s> base_span <s> rows_per_cta <r> stage_floats <f>
//                                              smem <b> kernel <k> ctas_per_sm <c>"
//   resample_shape list <pairs.i32> <out.i32>  one int32 row per (orig_freq, new_freq) pair: orig_freq, then the same
//                                              13 numbers
// kernel: -1 rejected (more than 4096 phases: SEPT_E_UNSUPPORTED), 0 simple, 1 tiled, 2 tiled with the unrolled
// 43-tap loop.  rows_per_cta, stage_floats and smem are the tiled kernel's, also for a pair that takes the simple one;
// ctas_per_sm is 0 there.  group_span: the widest spread of first stored taps among a group's phases; base_span:
// base_max - base_min over the groups.  Pairs are reduced by their gcd as sept_resample_f32 does.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include "resample_shape.h"
#include "tables.h"

using namespace sept;

static std::vector<int> shape_of(int orig_freq, int new_freq) {
    const int g = std::gcd(orig_freq, new_freq), orig = orig_freq / g, up = new_freq / g;
    if (orig > 4096 || up > 4096) return {orig, up, 0, 0, 0, 0, 0, 0, 0, 0, 0, -1, 0};
    std::vector<int32_t> k_lo;
    std::vector<float> rows;
    int taps = 0;
    const int width = make_resample_rows(orig, up, k_lo, rows, taps);
    ResampleTiles t;
    make_resample_tiles(up, taps, k_lo, rows, t);
    int group_span = 0;
    for (int j = 0; j < up; ++j)
        if (k_lo[j] - t.base[j / 4] > group_span) group_span = k_lo[j] - t.base[j / 4];
    const TileGeom geo = resample_tile_geom(orig, t.n_groups, t.tg, t.base_min, t.base_max);
    const size_t smem = resample_tiled_smem(orig, t.n_groups, t.tg, t.base_min, t.base_max);
    const ResampleShape s = resample_shape(true, orig, t.n_groups, t.tg, t.base_min, t.base_max);
    return {orig, up, width, taps, t.n_groups, t.tg, group_span, t.base_max - t.base_min, geo.rows_per_cta,
            geo.stage_floats, (int)smem, (int)s.kernel, s.ctas_per_sm};
}

static const char* const kNames[] = {"orig", "up", "width", "taps", "n_groups", "tg", "group_span", "base_span",
                                      "rows_per_cta", "stage_floats", "smem", "kernel", "ctas_per_sm"};

int main(int argc, char** argv) {
    if (argc == 4 && std::strcmp(argv[1], "list") == 0) {
        FILE* f = std::fopen(argv[2], "rb");
        if (!f) return 2;
        std::vector<int32_t> pairs;
        int32_t v[2];
        while (std::fread(v, sizeof(int32_t), 2, f) == 2) pairs.insert(pairs.end(), v, v + 2);
        std::fclose(f);
        std::vector<int32_t> out;
        for (size_t i = 0; i < pairs.size(); i += 2) {
            if (pairs[i] <= 0 || pairs[i + 1] <= 0) return 3;
            const std::vector<int> s = shape_of(pairs[i], pairs[i + 1]);
            out.push_back(pairs[i]);
            out.insert(out.end(), s.begin(), s.end());
        }
        f = std::fopen(argv[3], "wb");
        if (!f || std::fwrite(out.data(), sizeof(int32_t), out.size(), f) != out.size()) return 2;
        std::fclose(f);
        return 0;
    }
    if (argc != 3) return 1;
    const int orig_freq = std::atoi(argv[1]), new_freq = std::atoi(argv[2]);
    if (orig_freq <= 0 || new_freq <= 0) return 3;
    const std::vector<int> s = shape_of(orig_freq, new_freq);
    for (size_t i = 0; i < s.size(); ++i) std::printf("%s%s %d", i ? " " : "", kNames[i], s[i]);
    std::printf("\n");
    return 0;
}
