// Launch rule of the sinc resampler (resample.cu): the tiled kernel's rows per CTA and stage size, its shared memory,
// and which kernel a rate pair takes.  Host and device code, shared by the launcher, by the tiled kernel and by
// tests/hostsim/resample_shape.cpp, which reports the launch configuration of any rate pair.  Internal header.
#pragma once
#include <cuda_runtime.h>
#include <cstddef>

namespace sept {

constexpr int kTileThreads = 256;                      // threads of one half of a tiled CTA
constexpr int kTileTapsFast = 43;                      // taps of a 4-phase group at 44.1 -> 16 kHz (the reference's MSP-Improv case)
constexpr size_t kTiledMaxSmem = 112 * 1024;           // two CTAs per SM at least; larger tables take the simple kernel
constexpr size_t kTiled3CtaSmem = 72 * 1024;           // three CTAs per SM at or below this

struct TileGeom { int rows_per_cta, stage_floats; };

__host__ __device__ inline TileGeom resample_tile_geom(int orig, int n_groups, int tg, int base_min, int base_max) {
    // rows (m) per CTA: a multiple of 4, about kTileThreads tiles, and a stage of at most ~9k floats
    int mg = kTileThreads / n_groups;
    const int mg_fit = (9000 / orig - 4) / 4;
    if (mg > mg_fit) mg = mg_fit;
    if (mg < 1) mg = 1;
    TileGeom g;
    g.rows_per_cta = 4 * mg;
    // rows m_lo .. m_lo + 4 (mg + 1) - 1 can be touched (a CTA's sample range need not start on a row boundary)
    g.stage_floats = ((4 * (mg + 1) - 1) * orig + (base_max - base_min) + tg + 3 + 4) & ~3;   // + 3: 16-byte aligned fill
    return g;
}

// weight table, group bases and the two halves' stages
inline size_t resample_tiled_smem(int orig, int n_groups, int tg, int base_min, int base_max) {
    const TileGeom geo = resample_tile_geom(orig, n_groups, tg, base_min, base_max);
    return (size_t)n_groups * tg * 16 + (size_t)((n_groups + 3) & ~3) * 4 + 2 * (size_t)geo.stage_floats * 4;
}

enum ResampleKernel { kResampleSimple = 0, kResampleTiled = 1, kResampleTiledFast = 2 };   // resample_kernel, resample_tiled_kernel<0>, <kTileTapsFast>

struct ResampleShape {
    ResampleKernel kernel;
    TileGeom geo;          // tiled kernels only
    size_t smem;           // tiled kernels only
    int ctas_per_sm;       // resident CTAs per SM of a tiled kernel's persistent grid
};

// The kernel a rate pair with this register-tile table takes (has_tiles false: only the simple kernel is available).
inline ResampleShape resample_shape(bool has_tiles, int orig, int n_groups, int tg, int base_min, int base_max) {
    ResampleShape s{kResampleSimple, {0, 0}, 0, 0};
    if (!has_tiles) return s;
    const size_t smem = resample_tiled_smem(orig, n_groups, tg, base_min, base_max);
    if (smem > kTiledMaxSmem) return s;
    s.kernel = tg == kTileTapsFast ? kResampleTiledFast : kResampleTiled;
    s.geo = resample_tile_geom(orig, n_groups, tg, base_min, base_max);
    s.smem = smem;
    s.ctas_per_sm = smem <= kTiled3CtaSmem ? 3 : 2;
    return s;
}

}  // namespace sept
