// Launch configuration of the log-mel forward and backward for a shape (TEST CODE): computed with the library's own
// functions (tables.h: make_mel_program, extract_core.cuh: extract_mel_fast_ok, launch_shape.h: extract_warps,
// logmel_bwd_warps), so a test can name the kernel path a shape takes and notice when a tile change moves it.
//   launch_shape <n_fft> <hop> <n_mels>   prints "mel_fast <0|1> fwd_warps <w> bwd_warps <w> n_mel_entries <n>"
//   launch_shape sweep <out.i32>          writes int32 rows {n_fft, hop, mel_fast, fwd_warps, bwd_warps, n_mel_entries,
//                                         n_mels} for every n_fft of the C ABI, even hop <= n_fft and n_mels 1..512
// A warp count of 0 means the shape does not fit in shared memory.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "launch_shape.h"
#include "tables.h"

using namespace sept;

struct Shape { int mel_fast, fwd, bwd, entries; };

static Shape shape_of(int n_fft, int hop, int n_mels, const MelProgram& prog) {
    Shape s{};
    s.entries = (int)prog.entries.size();
    s.mel_fast = extract_mel_fast_ok(n_fft, n_mels, prog.n_head, prog.round_steps.data(), (int)prog.round_steps.size());
    switch (n_fft) {
        case 400: s.fwd = extract_warps<8>(hop, s.entries); s.bwd = logmel_bwd_warps<8>(hop, n_mels, s.entries); break;
        case 800: s.fwd = extract_warps<16>(hop, s.entries); s.bwd = logmel_bwd_warps<16>(hop, n_mels, s.entries); break;
        case 1600: s.fwd = extract_warps<32>(hop, s.entries); s.bwd = logmel_bwd_warps<32>(hop, n_mels, s.entries); break;
    }
    return s;
}

int main(int argc, char** argv) {
    if (argc == 3 && std::strcmp(argv[1], "sweep") == 0) {
        std::vector<int32_t> rows;
        for (int n_fft : {400, 800, 1600})
            for (int n_mels = 1; n_mels <= 512; ++n_mels) {
                MelProgram prog;
                make_mel_program(n_fft, n_mels, 16000, prog);
                for (int hop = 2; hop <= n_fft; hop += 2) {
                    const Shape s = shape_of(n_fft, hop, n_mels, prog);
                    rows.insert(rows.end(), {n_fft, hop, s.mel_fast, s.fwd, s.bwd, s.entries, n_mels});
                }
            }
        FILE* f = std::fopen(argv[2], "wb");
        if (!f || std::fwrite(rows.data(), sizeof(int32_t), rows.size(), f) != rows.size()) return 2;
        std::fclose(f);
        return 0;
    }
    if (argc != 4) return 1;
    const int n_fft = std::atoi(argv[1]), hop = std::atoi(argv[2]), n_mels = std::atoi(argv[3]);
    if ((n_fft != 400 && n_fft != 800 && n_fft != 1600) || hop <= 0 || hop > n_fft || (hop & 1) || n_mels < 1 || n_mels > 512)
        return 3;
    MelProgram prog;
    make_mel_program(n_fft, n_mels, 16000, prog);
    const Shape s = shape_of(n_fft, hop, n_mels, prog);
    std::printf("mel_fast %d fwd_warps %d bwd_warps %d n_mel_entries %d\n", s.mel_fast, s.fwd, s.bwd, s.entries);
    return 0;
}
