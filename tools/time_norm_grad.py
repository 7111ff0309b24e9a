#!/usr/bin/env python3
"""Time the gradient through per-speaker statistics and normalised training windows (normalization.speaker_stats_grad +
normalized_windows_grad) on the bench corpus (5531 utterances, ~9 audio-hours of log-mel at n_fft 800, 10 speakers round
robin, every training window; every input exceeds L2), with CUDA events after a warm-up: forward, backward with the
statistics differentiated and held constant, per-kernel times from torch.profiler, the bytes each kernel must move
(computed from shapes) against the HBM data-sheet bandwidth, and as a yardstick torch fp32 autograd of the same
computation (stacked rows per speaker, zero-padded window gather) on the same GPU in the same run.  Prints one JSON line;
with --out also writes it there."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
from oracle import norm_autograd
from speech_emotion_privacy_trust_b200 import extraction
from speech_emotion_privacy_trust_b200 import normalization as nz

HBM_TBPS = 7.7            # NVIDIA HGX B200 data sheet, per GPU
KERNELS = ("normalize_bwd_kernel", "normalize_bwd_merge_kernel", "stats_bwd_ties_kernel", "stats_bwd_tie_merge_kernel",
           "stats_bwd_frames_kernel")


def events_ms(fn, reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def kernel_ms(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for tag in KERNELS:
            if tag + "<" in e.key or tag + "(" in e.key:
                out[tag] = out.get(tag, 0.0) + e.device_time_total / 1000.0      # us -> ms
    return out


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
    feats, lay = extraction.logmel(batch, n_fft=800)
    del batch
    n_utts, F, TF = lay.frame_off_host.size - 1, feats.shape[1], lay.total_frames
    spk = [u % 10 for u in range(n_utts)]
    wu, wt = nz.window_table(lay)
    nw = len(wu)
    feat = feats.requires_grad_(True)
    G = torch.randn((nw, 1, 200, F), device=dev)

    def forward():
        st = nz.speaker_stats_grad(feat, lay, spk)
        return st, nz.normalized_windows_grad(feat, lay, st, wu, wt)

    st, win = forward()
    torch.autograd.grad(win, feat, G, retain_graph=True)                      # warm-up
    fwd = events_ms(forward, args.reps)
    bwd = events_ms(lambda: torch.autograd.grad(win, feat, G, retain_graph=True), args.reps)
    k_full = kernel_ms(lambda: torch.autograd.grad(win, feat, G, retain_graph=True))
    st_c = nz.speaker_stats(feat.detach(), lay, spk)
    win_c = nz.normalized_windows_grad(feat, lay, st_c, wu, wt)
    torch.autograd.grad(win_c, feat, G, retain_graph=True)
    bwd_c = events_ms(lambda: torch.autograd.grad(win_c, feat, G, retain_graph=True), args.reps)
    k_const = kernel_ms(lambda: torch.autograd.grad(win_c, feat, G, retain_graph=True))
    del win_c, st_c

    # bytes each kernel must move (fp32): Zbar once, features and dfeat once per pass
    fb, zb = TF * F * 4, nw * 200 * F * 4
    need = {"normalize_bwd_kernel": zb + 2 * fb, "stats_bwd_ties_kernel": fb, "stats_bwd_frames_kernel": 2 * fb}
    need_const = zb + fb
    kernels = {}
    for k, ms in k_full.items():
        row = {"ms": round(ms, 4)}
        if k in need:
            row.update(gb=round(need[k] / 1e9, 3), tb_per_s=round(need[k] / ms / 1e9, 2),
                       share_of_hbm=round(need[k] / ms / 1e9 / HBM_TBPS, 3))
        kernels[k] = row
    kc = k_const.get("normalize_bwd_kernel", float("nan"))

    # yardstick: torch fp32 autograd of the same computation, vectorised (one gather per speaker and one for windows)
    fo = lay.frame_off_host
    mult = np.concatenate([norm_autograd.stacked_rows(int(fo[u + 1] - fo[u])).numpy() + fo[u] for u in range(n_utts)])
    spk_rows = np.concatenate([np.full(len(norm_autograd.stacked_rows(int(fo[u + 1] - fo[u]))), spk[u]) for u in range(n_utts)])
    rows_of = [torch.from_numpy(mult[spk_rows == s]).to(dev) for s in range(10)]
    r = np.arange(200)
    idx = wt[:, None].astype(np.int64) + r[None, :]
    T_w = (fo[wu + 1] - fo[wu])[:, None]
    gidx = np.where(idx < T_w, fo[wu][:, None] + idx, TF)                    # TF: the appended zero row (padding)
    gidx = torch.from_numpy(gidx).to(dev)
    spk_w = torch.from_numpy(np.asarray(spk)[wu]).to(dev)
    x32 = feat.detach().clone().requires_grad_(True)

    def torch_fwd_bwd():
        stats = []
        for s in range(10):
            rows = x32.index_select(0, rows_of[s])
            mean = rows.mean(0)
            var = ((rows - mean) ** 2).mean(0)
            stats.append(torch.stack([mean, torch.sqrt(var)]))
        stats = torch.stack(stats)
        xp = torch.cat([x32, torch.zeros((1, F), device=dev)])
        w = (xp[gidx] - stats[spk_w, 0][:, None]) / (stats[spk_w, 1][:, None] + 1e-5)
        torch.autograd.grad(w, x32, G.view(nw, 200, F))

    torch_fwd_bwd()
    ref = events_ms(torch_fwd_bwd, max(1, args.reps // 2))
    line = json.dumps({
        "gpu": gpu, "audio_hours": round(hours, 3), "utterances": int(n_utts), "frames": int(TF), "windows": int(nw),
        "features_gb": round(fb / 1e9, 3), "windows_gb": round(zb / 1e9, 3), "weighted_rows_per_frame": round(len(mult) / TF, 3),
        "forward_ms": round(fwd, 3), "backward_ms": round(bwd, 3), "backward_const_stats_ms": round(bwd_c, 3),
        "fwd_plus_bwd_ms": round(fwd + bwd, 3), "backward_ms_per_audio_hour": round(bwd / hours, 4),
        "kernels": kernels,
        "const_stats_normalize_bwd_kernel": {"ms": round(kc, 4), "gb": round(need_const / 1e9, 3),
                                             "tb_per_s": round(need_const / kc / 1e9, 2)},
        "hbm_bound_tb_per_s": HBM_TBPS,
        "torch_fp32_autograd_fwd_bwd_ms": round(ref, 3),
    })
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
