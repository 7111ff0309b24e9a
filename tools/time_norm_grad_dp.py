#!/usr/bin/env python3
"""Time the data-parallel gradient through per-speaker statistics and normalised training windows
(normalization.speaker_stats_distributed_grad + normalized_windows_grad) under torchrun:

    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 --master-port 29581 \\
        tools/time_norm_grad_dp.py --out profiles/norm_grad_dp_nN.json

The bench corpus (5531 utterances, ~9 audio-hours, 10 speakers round robin) is split over the ranks with
parallel.shard_by_length, so every speaker has utterances on every rank.  Per rank, with CUDA events after a warm-up (every
timed region starts after a barrier): the forward (local statistics + all-gather + Chan merge + window gather) and its two
parts, speaker_stats_grad on the rank's utterances alone for scale, the backward with the statistics differentiated, and
the two exchanges of that backward on their own (the all-gather + rank-order sum of dstats, the int32 all-reduce of the
tie weights).  Rank 0 prints one JSON line with every rank's numbers and the card
name and power limit read in the same run; with --out it also writes it there."""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import bench
from speech_emotion_privacy_trust_b200 import extraction, parallel
from speech_emotion_privacy_trust_b200 import normalization as nz


def events_ms(fn, reps):
    dist.barrier()
    torch.cuda.synchronize()
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
    ap.add_argument("--out", help="rank 0 also writes the JSON result to this file")
    args = ap.parse_args()
    rank, local, world = bench.dist_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist.init_process_group("nccl", device_id=dev)
    try:
        gpu = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             stdout=subprocess.PIPE, text=True).stdout.strip()
        lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
        mine = parallel.shard_by_length(lengths, world)[rank]
        off = np.concatenate([[0], np.cumsum(lengths[mine])]).astype(np.int64)
        batch = extraction.RaggedAudio(bench.synth_corpus_device(lengths[mine], 4321 + rank, dev), off)
        feats, lay = extraction.logmel(batch, n_fft=800)
        del batch
        F = feats.shape[1]
        spk = [int(u) % 10 for u in mine]
        all_speakers = list(range(10))
        wu, wt = nz.window_table(lay)
        feat = feats.requires_grad_(True)
        G = torch.randn((len(wu), 1, 200, F), device=dev)

        def forward():
            st = nz.speaker_stats_distributed_grad(feat, lay, spk, all_speakers)
            return nz.normalized_windows_grad(feat, lay, st, wu, wt)

        win = forward()
        torch.autograd.grad(win, feat, G, retain_graph=True)                  # warm-up (NCCL communicators included)
        fwd = events_ms(forward, args.reps)
        st = nz.speaker_stats_distributed_grad(feat, lay, spk, all_speakers)
        fwd_stats = events_ms(lambda: nz.speaker_stats_distributed_grad(feat, lay, spk, all_speakers), args.reps)
        fwd_local = events_ms(lambda: nz.speaker_stats_grad(feat, lay, spk), args.reps)
        fwd_windows = events_ms(lambda: nz.normalized_windows_grad(feat, lay, st, wu, wt), args.reps)
        bwd = events_ms(lambda: torch.autograd.grad(win, feat, G, retain_graph=True), args.reps)
        dstats = torch.randn((10, 5, F), device=dev)
        ties = torch.ones((10, 2, F), dtype=torch.int32, device=dev)
        parallel.sum_in_rank_order(dstats, None)
        gather = events_ms(lambda: parallel.sum_in_rank_order(dstats, None), args.reps)
        reduce = events_ms(lambda: parallel.allreduce_exact_sum(ties, None), args.reps)
        mine_row = {"rank": rank, "gpu": gpu, "utterances": int(len(mine)), "frames": int(lay.total_frames),
                    "windows": int(len(wu)), "forward_ms": round(fwd, 3), "forward_stats_ms": round(fwd_stats, 3),
                    "forward_windows_ms": round(fwd_windows, 3), "local_speaker_stats_grad_ms": round(fwd_local, 3),
                    "backward_ms": round(bwd, 3),
                    "dstats_allgather_sum_ms": round(gather, 4), "ties_allreduce_ms": round(reduce, 4)}
        rows = [None] * world
        dist.all_gather_object(rows, mine_row)
        if rank == 0:
            line = json.dumps({
                "workload": "bench corpus (5531 utterances, 10 speakers) split by shard_by_length; "
                            "speaker_stats_distributed_grad -> normalized_windows_grad, every training window",
                "world_size": world, "audio_hours": round(float(lengths.sum()) / 16000 / 3600, 3),
                "gpus": sorted({r["gpu"] for r in rows}), "reps": args.reps,
                "max_forward_ms": max(r["forward_ms"] for r in rows), "max_backward_ms": max(r["backward_ms"] for r in rows),
                "ranks": rows,
            })
            print(line)
            if args.out:
                Path(args.out).parent.mkdir(parents=True, exist_ok=True)
                Path(args.out).write_text(line + "\n")
    finally:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
