// Warps per CTA of the extraction forward (extract.cu) and of the log-mel backward's frame pass (extract_bwd.cu): as
// many warp tiles as fit beside the CTA constants in shared memory.  Host code, shared by the launchers and by
// tests/hostsim/launch_shape.cpp, which reports the launch configuration of any (n_fft, hop, n_mels).  Internal header.
#pragma once
#include "extract.h"
#include "extract_bwd.cuh"

namespace sept {

constexpr size_t kExtractMaxSmem = kMaxDynSmem - 64;  // minus the forward's static shared memory (tmem_base, cta_next)

// forward: 0 when not even one warp fits (the C ABI refuses such a shape)
template <int R>
inline int extract_warps(int hop, int n_mel_entries) {
    using G = Geo<R>;
    return warps_that_fit(extract_const_bytes(R, n_mel_entries), G::stage_floats(hop) * 4 + G::Y_PK4 * 16,
                          ExtractWarps<R>::value, kExtractMaxSmem);
}

// backward frame pass: its warp tiles add the mel sums U, D of n_mels bands to the forward's
template <int R>
inline int logmel_bwd_warps(int hop, int n_mels, int n_mel_entries) {
    return warps_that_fit(extract_const_bytes(R, n_mel_entries), Bwd<Geo<R>>::warp_floats(hop, n_mels) * 4, kBwdWarps,
                          kMaxDynSmem);
}

}  // namespace sept
