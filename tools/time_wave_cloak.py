#!/usr/bin/env python3
"""Time the waveform-domain cloak (wave_cloak.WaveCloak, period 32 000) on the bench corpus (5531 utterances, ~9.2
audio-hours, ~532 M samples: x, y and the gradient each exceed L2), with CUDA events after a warm-up: the forward (noise
draw + wave_add_kernel) and the backward (wave_reduce_kernel + wave_merge_kernel + the mu / rho kernel), per-kernel times
from torch.profiler, and the bytes each must move, computed from shapes, against the HBM data-sheet bandwidth.  In the
same run, the same for per-utterance noise (WaveCloak(per_utterance=True): wave_sigma_kernel + wave_eval_add_kernel
forward, wave_reduce_per_utt_kernel + wave_merge_per_utt_kernel backward), under "per_utterance".  The card's name and
power limit are read in the same run.  Prints one JSON line; with --out also writes it there."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
from speech_emotion_privacy_trust_b200 import extraction, wave_cloak

HBM_TBPS = 7.7            # NVIDIA HGX B200 data sheet, per GPU
KERNELS = ("wave_add_kernel", "wave_reduce_kernel", "wave_merge_kernel", "cloak_fwd_kernel", "cloak_bwd_kernel",
           "wave_sigma_kernel", "wave_eval_add_kernel", "wave_reduce_per_utt_kernel", "wave_merge_per_utt_kernel")


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_ms(fn, reps):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for tag in KERNELS:
            if tag + "(" in e.key or tag + "<" in e.key:
                out[tag] = out.get(tag, 0.0) + e.device_time_total / 1000.0 / reps      # us -> ms per call
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--period", type=int, default=wave_cloak.DEFAULT_PERIOD)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_wave_cloak.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(bench.synth_corpus_device(lengths, 4321, dev), off)
    n, L = batch.wav.numel(), args.period
    hours = float(n) / 16000 / 3600
    layer = wave_cloak.WaveCloak(1e-4, 1e-2, period=L).to(dev)
    G = torch.randn(n, device=dev)

    def forward():
        return layer(batch).wav

    y = forward()
    y.backward(G, retain_graph=True)                                          # warm-up (tiles, workspaces, modules)
    fwd = events_ms(forward, args.reps)
    bwd = events_ms(lambda: y.backward(G, retain_graph=True), args.reps)
    k = kernel_ms(forward, args.reps)
    k.update(kernel_ms(lambda: y.backward(G, retain_graph=True), args.reps))

    ws_rows = wave_cloak._lib.lib().sept_wave_cloak_bwd_workspace_bytes(L)
    table = 8 * (batch.n_utts + 1)
    need = {                                                                  # bytes each kernel must move (fp32)
        "wave_add_kernel": 8 * n + table + 4 * L,                             # x read, y written, offsets, noise
        "wave_reduce_kernel": 4 * n + 2 * table + ws_rows,                    # g read, offsets + tiles, partial rows written
        "wave_merge_kernel": ws_rows + 4 * L,
    }

    pu = wave_cloak.WaveCloak(1e-4, 1e-2, period=L, per_utterance=True).to(dev)

    def forward_pu():
        return pu(batch).wav

    y_pu = forward_pu()
    y_pu.backward(G, retain_graph=True)                                       # warm-up
    fwd_pu = events_ms(forward_pu, args.reps)
    bwd_pu = events_ms(lambda: y_pu.backward(G, retain_graph=True), args.reps)
    k_pu = kernel_ms(forward_pu, args.reps)
    k_pu.update(kernel_ms(lambda: y_pu.backward(G, retain_graph=True), args.reps))
    ws_pu = wave_cloak._lib.lib().sept_wave_cloak_bwd_per_utt_workspace_bytes(L)
    need.update({
        "wave_eval_add_kernel": 8 * n + table + 8 * L,                        # x read, y written, offsets, mu and sigma
        "wave_reduce_per_utt_kernel": 4 * n + 2 * table + ws_pu,              # g read, offsets + tiles, both row sets written
        "wave_merge_per_utt_kernel": ws_pu + 12 * L,                          # both row sets, rho read, dlocs / drhos written
    })

    def rows(ks):
        out = {}
        for name, ms in ks.items():
            row = {"ms": round(ms, 4)}
            if name in need:
                row.update(gb=round(need[name] / 1e9, 3), gb_per_s=round(need[name] / ms / 1e6, 1),
                           share_of_hbm=round(need[name] / ms / 1e9 / HBM_TBPS, 3))
            out[name] = row
        return out

    kernels = rows(k)
    fwd_bytes, bwd_bytes = 8 * n + table, 4 * n
    line = json.dumps({
        "gpu": gpu, "period": L, "audio_hours": round(hours, 3), "utterances": int(batch.n_utts), "samples": int(n),
        "tiles": batch.tiles(L).n_tiles, "forward_ms": round(fwd, 3), "backward_ms": round(bwd, 3),
        "forward_audio_hours_per_s": round(hours / fwd * 1e3, 1), "backward_audio_hours_per_s": round(hours / bwd * 1e3, 1),
        "forward_gb": round(fwd_bytes / 1e9, 3), "backward_gb": round(bwd_bytes / 1e9, 3),
        "forward_gb_per_s": round(fwd_bytes / fwd / 1e6, 1), "backward_gb_per_s": round(bwd_bytes / bwd / 1e6, 1),
        "kernels": kernels, "hbm_bound_tb_per_s": HBM_TBPS,
        "per_utterance": {"forward_ms": round(fwd_pu, 3), "backward_ms": round(bwd_pu, 3), "kernels": rows(k_pu),
                          "backward_workspace_gb": round(ws_pu / 1e9, 4)},
    })
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
