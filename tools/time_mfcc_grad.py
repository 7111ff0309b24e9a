#!/usr/bin/env python3
"""Time the MFCC waveform gradient (extraction.mfcc_grad) over the bench corpus (5531 utterances, ~9 audio-hours, larger
than L2), with CUDA events after a warm-up: forward, backward, its per-kernel split by torch.profiler (power recompute,
head, route, the two frame passes, gather), workspace bytes, and as a yardstick the same gradient from torch fp32
autograd through torch.stft, a torch np.gradient, per-utterance amax and the DCT, on the same GPU in the same run.
Prints one JSON line; with --out also writes it there."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
from oracle import restate
from speech_emotion_privacy_trust_b200 import _lib, extraction

KERNELS = {"recompute_power": "extract_kernel", "head": "mfcc_bwd_head_kernel", "route": "mfcc_bwd_route_kernel",
           "frame_pass_x": "logmel_bwd_frames_kernel<8, 0>", "frame_pass_grad": "logmel_bwd_frames_kernel<8, 1>",
           "gather": "mfcc_bwd_gather_kernel"}


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def np_gradient_rows(x, spacing):
    return torch.cat([(x[:, 1:2] - x[:, 0:1]) / spacing, (x[:, 2:] - x[:, :-2]) / (2.0 * spacing),
                      (x[:, -1:] - x[:, -2:-1]) / spacing], dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                         text=True).stdout.strip().splitlines()[0]
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(bench.synth_corpus_device(lengths, 4321, dev), off)
    hours = float(lengths.sum()) / 16000 / 3600
    lib = _lib.lib()
    lay = batch.layout(400, 200)
    G = torch.randn(lay.total_frames * 120, device=dev)
    wav = batch.wav.detach().requires_grad_(True)
    batch.wav = wav
    feats, _ = extraction.mfcc_grad(batch)
    torch.autograd.grad(feats, wav, G)                           # warm-up: modules, constants, allocator
    fwd = events_ms(lambda: extraction.mfcc(batch), args.reps)
    feats, _ = extraction.mfcc_grad(batch)
    bwd = events_ms(lambda: torch.autograd.grad(feats, wav, G, retain_graph=True), args.reps)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        torch.autograd.grad(feats, wav, G, retain_graph=True)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        for name, tag in KERNELS.items():
            if tag in e.key:
                kern[name] = kern.get(name, 0.0) + e.device_time_total / 1000.0   # us -> ms
    ws_bytes = int(lib.sept_mfcc_bwd_workspace_bytes(batch.n_utts, lay.total_frames, lay.n_items))

    # yardstick: torch fp32 autograd through the same chain, utterances zero-padded into chunks of 256
    fb = torch.from_numpy(restate.melscale_fbanks_htk(201, 128, dtype=np.float32)).to(dev)
    dct = torch.from_numpy(restate.create_dct_ortho(40, 128, np.float32)).to(dev)
    win = torch.hann_window(400, device=dev)
    chunks = []
    for c0 in range(0, len(lengths), 256):
        c1 = min(len(lengths), c0 + 256)
        L = int(lengths[c0:c1].max())
        x = torch.zeros(c1 - c0, L, device=dev)
        for i in range(c0, c1):
            x[i - c0, :lengths[i]] = wav.detach()[off[i]:off[i + 1]]
        chunks.append(x.requires_grad_(True))

    def torch_fwd_bwd():
        for x in chunks:
            outs = []
            for y in (x, np_gradient_rows(x, 1.0), np_gradient_rows(x, 2.0)):
                X = torch.stft(y, 400, 200, window=win, center=True, pad_mode="reflect", return_complex=True)
                M = (X.real * X.real + X.imag * X.imag).transpose(1, 2) @ fb
                D = 10.0 * torch.log10(torch.clamp(M, min=1e-10))
                F = torch.maximum(D, D.amax(dim=(1, 2), keepdim=True) - 80.0)
                outs.append(F @ dct)
            out = torch.cat(outs, dim=2)
            torch.autograd.grad(out, x, torch.ones_like(out))

    torch_fwd_bwd()
    ref = events_ms(torch_fwd_bwd, max(1, args.reps // 2))
    result = {
        "gpu": gpu, "audio_hours": round(hours, 3), "utterances": int(len(lengths)), "frames": lay.total_frames,
        "forward_ms": round(fwd, 3), "backward_ms": round(bwd, 3),
        "forward_ms_per_audio_hour": round(fwd / hours, 4), "backward_ms_per_audio_hour": round(bwd / hours, 4),
        "backward_kernels_ms": {k: round(kern.get(k, float("nan")), 3) for k in KERNELS},
        "backward_kernels_ms_per_audio_hour": {k: round(kern.get(k, float("nan")) / hours, 4) for k in KERNELS},
        "workspace_bytes": ws_bytes, "workspace_gb_per_audio_hour": round(ws_bytes / 1e9 / hours, 3),
        "torch_fp32_autograd_fwd_bwd_ms": round(ref, 3), "torch_fp32_autograd_ms_per_audio_hour": round(ref / hours, 4),
        "ours_fwd_plus_bwd_ms": round(fwd + bwd, 3),
    }
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
