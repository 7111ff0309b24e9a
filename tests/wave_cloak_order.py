"""Host restatement of the waveform-cloak backward's summation order (csrc/wave_cloak.cu, DESIGN 3.3b), in float32 with
the kernels' additions one by one, so a test can hold the GPU result to it bit for bit and check its error against a
float64 sum.  Not a test module: test_wave_cloak_cpu.py and test_wave_cloak_gpu.py import it."""
import numpy as np

THREADS, SLICES, MERGE_LANES = 256, 592, 8          # kWaveThreads, kWaveSlices, kWaveMergeLanes (csrc/wave_cloak.h)


def tiles_of(utt_off, tile_off, period):
    """(base, length) of every tile, in tile order: tile k of utterance u starts at utt_off[u] + k * period."""
    utt_off, tile_off = np.asarray(utt_off, np.int64), np.asarray(tile_off, np.int64)
    u = np.repeat(np.arange(len(utt_off) - 1), np.diff(tile_off))
    base = utt_off[u] + (np.arange(int(tile_off[-1])) - tile_off[u]) * period
    return base, np.minimum(period, utt_off[u + 1] - base)


def phase_sum(g, utt_off, tile_off, period):
    """r[j]: g summed over every in-utterance sample of phase j, in the order of wave_reduce_kernel + wave_merge_kernel."""
    g = np.asarray(g, np.float32)
    base, length = tiles_of(utt_off, tile_off, period)
    n_tiles = len(base)
    rows = np.zeros((n_tiles, period), np.float32)             # tile t's samples by phase, +0 past the utterance's end
    for t in range(n_tiles):
        rows[t, :length[t]] = g[base[t]:base[t] + length[t]]
    q = period // 4
    lanes = 1 if q >= THREADS else THREADS // q
    partial = np.zeros((SLICES, period), np.float32)
    for s in range(SLICES):
        t0, t1 = n_tiles * s // SLICES, n_tiles * (s + 1) // SLICES
        acc = np.zeros(period, np.float32)
        for c0 in range(t0, t1, THREADS):
            chunk = rows[c0:min(c0 + THREADS, t1)]
            pad = -len(chunk) % lanes                          # lane l takes the chunk's tiles l, l + lanes, ...
            chunk = np.concatenate([chunk, np.zeros((pad, period), np.float32)]).reshape(-1, lanes, period)
            lane = np.zeros((lanes, period), np.float32)
            for i in range(chunk.shape[0]):
                lane = lane + chunk[i]
            c = lane[0]
            for k in range(1, lanes):
                c = c + lane[k]
            acc = acc + c
        partial[s] = acc
    per = SLICES // MERGE_LANES
    merged = []
    for k in range(MERGE_LANES):
        a = np.zeros(period, np.float32)
        for s in range(k * per, (k + 1) * per):
            a = a + partial[s]
        merged.append(a)
    r = merged[0]
    for k in range(1, MERGE_LANES):
        r = r + merged[k]
    return r


def phase_of(utt_off, n, period):
    """Per sample of an n-sample buffer: its phase, or -1 outside every utterance."""
    utt_off = np.asarray(utt_off, np.int64)
    ph = np.full(n, -1, np.int64)
    for u in range(len(utt_off) - 1):
        a, b = int(utt_off[u]), int(utt_off[u + 1])
        ph[a:b] = np.arange(b - a) % period
    return ph


def bound(g, utt_off, period):
    """(float64 phase sums, per-phase bound 4 * 2^-23 * sqrt(n_j) * sum |g| over phase j)."""
    ph = phase_of(utt_off, len(g), period)
    inside = ph >= 0
    g64 = np.asarray(g, np.float64)[inside]
    r64 = np.bincount(ph[inside], weights=g64, minlength=period)
    n_j = np.bincount(ph[inside], minlength=period)
    a_j = np.bincount(ph[inside], weights=np.abs(g64), minlength=period)
    return r64, 4 * 2.0 ** -23 * np.sqrt(n_j) * a_j
