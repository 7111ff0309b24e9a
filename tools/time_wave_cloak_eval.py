#!/usr/bin/env python3
"""Time the waveform cloak's per-utterance evaluation on the bench corpus (5531 utterances, ~9.2 audio-hours, ~532 M
samples, L = 32 000; x and y each exceed L2), with CUDA events after a warm-up, in one run:
  - sept_wave_cloak_eval_f32 (WaveCloak.noisy_per_utterance: sigma pre-pass + wave_eval_add_kernel + counter add), with
    the bytes it must move computed from shapes against the HBM data-sheet bandwidth;
  - wave_add_kernel (sept_wave_cloak_fwd_f32, one noise shared by every utterance) on the same batch: what the inline draw
    costs;
  - the torch composition a user would write without the fused entry: per-utterance noise rows from
    sept_cloak_fwd_f32(per_sample = 1) and an indexed add through a precomputed int64 (sample -> row element) index;
  - evaluation.wave_cloak_evaluate with the stock two_d_cnn_lstm pair, whole and broken down into noise, log-mel,
    statistics, window gather and classifiers.
Per-kernel times come from torch.profiler in separate passes.  The card's name and power limit are read in the same run.
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
from speech_emotion_privacy_trust_b200 import _lib, cloak_ops, evaluation, extraction, normalization, wave_cloak

HBM_TBPS = 7.7            # NVIDIA HGX B200 data sheet, per GPU
KERNELS = ("wave_eval_add_kernel", "wave_sigma_kernel", "wave_add_kernel", "cloak_fwd_kernel")


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


def hbm(nbytes, ms):
    return {"ms": round(ms, 4), "gb": round(nbytes / 1e9, 3), "gb_per_s": round(nbytes / ms / 1e6, 1),
            "share_of_hbm": round(nbytes / ms / 1e9 / HBM_TBPS, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--eval-reps", type=int, default=2)
    ap.add_argument("--period", type=int, default=wave_cloak.DEFAULT_PERIOD)
    ap.add_argument("--out", help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_wave_cloak_eval.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda", 0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(bench.synth_corpus_device(lengths, 4321, dev), off)
    n, L, U = batch.wav.numel(), args.period, batch.n_utts
    hours = float(n) / 16000 / 3600
    torch.manual_seed(0)
    layer = wave_cloak.WaveCloak(1e-4, 1e-2, period=L, locs=1e-3 * torch.randn(L)).to(dev)
    locs, rhos = layer.locs.detach(), layer.rhos.detach()
    res = {"gpu": gpu, "period": L, "audio_hours": round(hours, 3), "utterances": U, "samples": int(n),
           "unaligned_utterance_starts": int(np.count_nonzero(off[:-1] % 4)), "hbm_bound_tb_per_s": HBM_TBPS}

    # ---- the noise alone: fused entry, shared-noise add, torch composition -----------------------------------------
    def fused():
        return layer.noisy_per_utterance(batch)

    noise = torch.randn(L, device=dev) * 1e-2
    y_add = torch.empty_like(batch.wav)

    def add_only():
        _lib.launch("sept_wave_cloak_fwd_f32", batch.wav, batch.utt_off, U, n, noise, L, y_add, device=dev)

    zeros = torch.zeros(U * L, device=dev)
    utt = torch.repeat_interleave(torch.arange(U, device=dev), torch.from_numpy(lengths).to(dev))
    index = utt * L + (torch.arange(n, device=dev) - batch.utt_off[utt]) % L       # 8 B per sample, built once
    counter = torch.zeros(1, dtype=torch.int64, device=dev)

    def composed():
        rows, _, _ = cloak_ops.cloak_forward_raw(zeros, locs, rhos, None, None, torch.initial_seed(), 0, wave_cloak.EPS_STD,
                                                 layer.min_scale, layer.max_scale, draw=counter, per_sample=True)
        return batch.wav + rows[index]

    for fn in (fused, add_only, composed):
        fn()
    torch.cuda.synchronize()
    counter.zero_()
    layer._draws.zero_()
    same = torch.equal(fused().wav, composed())                                    # the two compute the same bits
    t_fused, t_add, t_comp = events_ms(fused, args.reps), events_ms(add_only, args.reps), events_ms(composed, args.reps)
    k_fused, k_add, k_comp = kernel_ms(fused, args.reps), kernel_ms(add_only, args.reps), kernel_ms(composed, args.reps)
    table = 8 * (U + 1)
    fused_bytes = 8 * n + table + 4 * 4 * L            # x read, y written, offsets; rhos + sigma + locs (+ sigma write)
    comp_bytes = 4 * U * L * 2 + 4 * U * L + 8 * n + 4 * n * 2       # zeros read + rows written, rows / index / x read, y
    del index, utt, zeros
    res.update({
        "fused_call_ms": round(t_fused, 3), "fused_audio_hours_per_s": round(hours / t_fused * 1e3, 1),
        "wave_eval_add_kernel": hbm(fused_bytes, k_fused.get("wave_eval_add_kernel", float("nan"))),
        "wave_sigma_kernel_ms": round(k_fused.get("wave_sigma_kernel", float("nan")), 4),
        "shared_noise_add_call_ms": round(t_add, 3),
        "wave_add_kernel": hbm(8 * n + table + 4 * L, k_add.get("wave_add_kernel", float("nan"))),
        "composition_ms": round(t_comp, 3), "composition_gb": round(comp_bytes / 1e9, 3),
        "composition_cloak_fwd_kernel_ms": round(k_comp.get("cloak_fwd_kernel", float("nan")), 4),
        "composition_index_gb_not_timed": round(8 * n / 1e9, 3),
        "fused_equals_composition": bool(same), "speedup_vs_composition": round(t_comp / t_fused, 2),
    })

    # ---- the whole evaluator, and its stages ---------------------------------------------------------------------
    from speech_emotion_privacy_trust_b200.dropin import baseline_models
    torch.manual_seed(8)
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0).to(dev).eval()
    base, adv = mk("emotion"), mk("gender")
    spk = [f"s{u % 10}" for u in range(U)]                                         # ten speakers
    max_windows = 512

    def whole():
        return evaluation.wave_cloak_evaluate(layer, base, adv, batch, speaker_of_utt=spk, max_windows=max_windows)

    whole()
    t_whole = events_ms(whole, args.eval_reps)
    stage = {}

    def timed(name, fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        stage[name] = round(stage.get(name, 0.0) + a.elapsed_time(b) / args.eval_reps, 3)
        return out

    for _ in range(args.eval_reps):
        noisy = timed("noise_ms", fused)
        feat, lay = timed("logmel_ms", lambda: extraction.logmel(noisy))
        st = timed("stats_ms", lambda: normalization.speaker_stats(feat, lay, spk, whole_utterance=[True] * U))
        wu, wt = evaluation.eval_window_table(lay)
        chunks = timed("window_gather_ms", lambda: [normalization.normalized_windows(feat, lay, st, wu[a:a + max_windows],
                                                                                     wt[a:a + max_windows])
                                                    for a in range(0, len(wu), max_windows)])

        def classify():
            with torch.no_grad():
                for x in chunks:
                    torch.softmax(base(x), 1)
                    torch.softmax(adv(x), 1)

        timed("classifiers_ms", classify)
        del chunks
    res.update({"evaluate_ms": round(t_whole, 2), "evaluate_windows": int(len(wu)), "evaluate_max_windows": max_windows,
                "evaluate_stages": stage, "classifiers": "two_d_cnn_lstm h=64 (emotion, gender), fp32, TF32 at torch defaults"})
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
