#!/usr/bin/env python3
"""Time the log-mel waveform gradient (extraction.logmel_grad) over the bench corpus (5531 utterances, ~9 audio-hours,
larger than L2), with CUDA events after a warm-up: forward, backward (frame pass + gather pass, split by torch.profiler
kernel times), workspace bytes, and as a yardstick the same gradient from torch autograd over torch.stft (cuFFT) on the
same GPU in the same run.  Prints one JSON line; with --out also writes it there."""
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


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


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
    result = {"gpu": gpu, "audio_hours": round(hours, 3), "utterances": int(len(lengths))}
    for n_fft in (800, 1600):
        hop = 160
        lay = batch.layout(n_fft, hop)
        G = torch.randn(lay.total_frames, 128, device=dev)
        wav = batch.wav.detach().requires_grad_(True)
        batch.wav = wav
        feats, _ = extraction.logmel_grad(batch, n_fft=n_fft, hop=hop)
        torch.autograd.grad(feats, wav, G)                       # warm-up: modules, constants, allocator
        fwd = events_ms(lambda: extraction.logmel(batch, n_fft=n_fft, hop=hop), args.reps)
        feats, _ = extraction.logmel_grad(batch, n_fft=n_fft, hop=hop)
        bwd = events_ms(lambda: torch.autograd.grad(feats, wav, G, retain_graph=True), args.reps)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            torch.autograd.grad(feats, wav, G, retain_graph=True)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            for tag in ("logmel_bwd_frames_kernel", "logmel_bwd_gather_kernel"):
                if tag in e.key:
                    kern[tag] = kern.get(tag, 0.0) + e.device_time_total / 1000.0   # us -> ms
        # yardstick: torch autograd through torch.stft on the same corpus, utterances zero-padded into chunks of 256
        fb = torch.from_numpy(restate.melscale_fbanks_htk(n_fft // 2 + 1, 128, dtype=np.float32)).to(dev)
        win = torch.hann_window(n_fft, device=dev)
        chunks = []
        for c0 in range(0, len(lengths), 256):
            c1 = min(len(lengths), c0 + 256)
            L = int(lengths[c0:c1].max())
            x = torch.zeros(c1 - c0, L, device=dev)
            for i in range(c0, c1):
                x[i - c0, :lengths[i]] = batch.wav.detach()[off[i]:off[i + 1]]
            chunks.append(x.requires_grad_(True))

        def torch_fwd_bwd():
            for x in chunks:
                X = torch.stft(x, n_fft, hop, window=win, center=True, pad_mode="reflect", return_complex=True)
                M = (X.real * X.real + X.imag * X.imag).transpose(1, 2) @ fb
                D = 10.0 * torch.log10(torch.clamp(M, min=1e-10))
                torch.autograd.grad(D, x, torch.ones_like(D))

        torch_fwd_bwd()
        ref = events_ms(torch_fwd_bwd, max(1, args.reps // 2))
        result[f"n_fft_{n_fft}"] = {
            "forward_ms": round(fwd, 3), "backward_ms": round(bwd, 3),
            "frame_pass_ms": round(kern.get("logmel_bwd_frames_kernel", float("nan")), 3),
            "gather_pass_ms": round(kern.get("logmel_bwd_gather_kernel", float("nan")), 3),
            "forward_ms_per_audio_hour": round(fwd / hours, 4), "backward_ms_per_audio_hour": round(bwd / hours, 4),
            "workspace_bytes": int(lib.sept_logmel_bwd_workspace_bytes(n_fft, hop, lay.n_items)),
            "workspace_gb_per_audio_hour": round(lib.sept_logmel_bwd_workspace_bytes(n_fft, hop, lay.n_items) / 1e9 / hours, 3),
            "torch_stft_autograd_fwd_bwd_ms": round(ref, 3),
            "torch_stft_autograd_ms_per_audio_hour": round(ref / hours, 4),
            "ours_fwd_plus_bwd_ms": round(fwd + bwd, 3),
        }
        del chunks, feats, G
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
