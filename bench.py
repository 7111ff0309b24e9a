#!/usr/bin/env python3
"""bench.py -- the headline metric of BASELINE.json on synthetic data: log-mel audio-hours/sec (n_fft 800, hop 160,
128 mels) over an IEMOCAP-sized corpus, plus cloak+GRL training utterances/sec as a secondary figure.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

One step = one pass of the extraction hot path over one corpus-sized ragged batch (5531 utterances, 2-10 s each,
~9.2 audio-hours, 2.1 GB of fp32 waveform -- larger than the 126 MB L2, so no flush is needed between steps).
N > 1 (torchrun, one rank per GPU): ONE corpus of N x 5531 utterances is length-bucketed and dealt to the ranks by
parallel.shard_by_length (every rank gets the same mix of lengths and the same amount of audio), no data-path collective
("scaling": "weak": the audio per GPU is fixed); the time is the max over ranks of the CUDA-event time of the K steps.

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for how each field is obtained.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

N_FFT, HOP, N_MELS = 800, 160, 128
E2E_PCM16_MS = None
CORPUS_UTTS = 5531                         # IEMOCAP 4-class size (SURVEY 8d, config 1)
FLOP_PER_FRAME = 22999                     # BASELINE.md section 3: log-mel n_fft=800 (rFFT 2.5 N log2 N + window + power + mel + log)
BYTES_PER_FRAME = 4 * HOP + 4 * N_MELS     # waveform read once + features written once = 1152 B
FP32_LANES_PER_SM = 128
DUMP_ROWS = 65536                          # feature rows --dump-outputs writes, split over the ranks: 32 MiB in all


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    return rank, local, world


def corpus_lengths(n_utts: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return rng.integers(2 * 16000, 10 * 16000 + 1, size=n_utts).astype(np.int64)


def synth_corpus_device(lengths: np.ndarray, seed: int, device, chunk: int = 128) -> torch.Tensor:
    """Speech-shaped synthetic audio generated on the device (workload generation, outside every timed region):
    white noise -> 1/sqrt(f) tilt -> 3-5 Hz syllabic envelope -> peak 0.3, per utterance (SURVEY 8d).  Utterances are
    made `chunk` at a time as rows of one padded matrix (torch.fft is used here only to MAKE the input signal)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    wav = torch.empty(int(lengths.sum()), dtype=torch.float32, device=device)
    pos = 0
    for c0 in range(0, len(lengths), chunk):
        lens = torch.as_tensor(lengths[c0:c0 + chunk], device=device)
        n = int(lens.max())
        n += n & 1
        white = torch.randn((len(lens), n), generator=g, device=device)
        f = torch.fft.rfftfreq(n, 1.0 / 16000, device=device)
        tilt = torch.where(f > 0, torch.rsqrt(torch.clamp(f, min=1e-6)), torch.zeros_like(f))
        x = torch.fft.irfft(torch.fft.rfft(white, dim=1) * tilt, n, dim=1)
        fm = 3.0 + 2.0 * torch.rand((len(lens), 1), generator=g, device=device)
        ph = 6.2831853 * torch.rand((len(lens), 1), generator=g, device=device)
        t = torch.arange(n, device=device, dtype=torch.float32) / 16000.0
        x = x * (0.5 * (1.0 + torch.sin(6.2831853 * fm * t + ph)))
        live = torch.arange(n, device=device)[None, :] < lens[:, None]
        x = x * live
        x = x * (0.3 / x.abs().amax(dim=1, keepdim=True).clamp_min(1e-12))
        total = int(lens.sum())
        wav[pos:pos + total] = x[live]
        pos += total
        del white, x, live
    return wav


class ClockSampler:
    """SM clock and throttle reasons sampled every ~5 ms through NVML while the timed region runs (the nvidia-smi query of
    B200_PROFILING.md cannot sample faster than its process start-up; NVML reads the same counters)."""
    REASONS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.rows, self.stop_flag, self.thread, self.nvml = [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.nvml = None

    @staticmethod
    def _physical_index(index: int) -> int:
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v for v in vis.split(",") if v.strip()]
            if index < len(ids) and ids[index].strip().isdigit():
                return int(ids[index])
        return index

    def _pump(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((time.perf_counter(), mhz, bits))
            except Exception:
                pass
            time.sleep(0.005)

    def window(self, t0, t1):
        rows = [r for r in self.rows if t0 <= r[0] <= t1] or self.rows[-3:]
        sm = [r[1] for r in rows]
        reasons = sorted(name for name, bit in self.REASONS.items() if any(r[2] & bit for r in rows))
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": getattr(self, "max_mhz", None),
                "reasons": reasons, "samples": len(sm), "source": "nvml"}

    def stop(self):
        self.stop_flag = True


def profiled_traffic(frames: int):
    """DRAM bytes per launch of the extraction kernel from the committed ncu capture (profiles/), scaled per frame when
    the workload size differs; None if no capture is committed."""
    cands = sorted((REPO / "profiles").glob("extract800_traffic_r*.json"))
    if N_FFT != 800 or not cands:
        return None
    t = json.loads(cands[-1].read_text())                       # the newest capture; regenerate it whenever extract.cu changes
    return int((t["dram_bytes_read"] + t["dram_bytes_write"]) * frames / t["frames"])


def measured_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return json.loads(p.read_text()), "measured"
        except ValueError:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


# --------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port of the reference's CPU path (oracle/ref_port.py, torchaudio)
# --------------------------------------------------------------------------------------------------------------
def cpu_sample_waves(n_utts: int, seed: int):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(seed)
    lens = corpus_lengths(n_utts, seed)
    return [torch.from_numpy(synth.speech_shaped(int(n), rng))[None] for n in lens]


def time_cpu_reference(waves, threads: int) -> float:
    """Seconds for one pass of the reference's per-utterance loop (audio_feature_extraction.py:180-186, mel1 only)."""
    from oracle import ref_port
    torch.set_num_threads(threads)
    t0 = time.perf_counter()
    for a in waves:
        ref_port.mel_spectrogram(a, n_fft=N_FFT, feature_len=N_MELS)
    return time.perf_counter() - t0


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n_sample = 240                                  # ~0.4 audio-hours per step: about a second of CPU work
    waves = cpu_sample_waves(n_sample, 1234)
    hours = sum(a.shape[1] for a in waves) / 16000 / 3600
    for _ in range(args.warmup):
        time_cpu_reference(waves, threads)
    t = [time_cpu_reference(waves, threads) for _ in range(args.steps)]
    total = sum(t)
    value = hours * args.steps / total
    sample = f"{n_sample} utterances ({hours:.3f} audio-h) of the seed-1234 corpus per step, one utterance per call"
    print(json.dumps({
        "impl": "reference", "metric": "log-mel audio-hours/sec", "value": value, "unit": "audio-hours/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(world, note="reference arm: bounded sample of the same workload on the host cores"),
        "cpu_baseline": {"value": value, "unit": "audio-hours/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "audio-hours/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def workload_config(world: int, note: str | None = None):
    cfg = {"workload": f"log-mel n_fft={N_FFT} hop={HOP} n_mels={N_MELS} (mel_spectrogram, mel1) over a synthetic "
                       f"IEMOCAP-sized corpus: {CORPUS_UTTS} utterances of 2-10 s at 16 kHz per GPU (BASELINE.json configs[0] "
                       "shape, batched as in configs[3])",
           "utterances_per_gpu": CORPUS_UTTS, "n_fft": N_FFT, "hop": HOP, "n_mels": N_MELS,
           "layout": "frame-major (T,128) per utterance",
           "sharding": f"one corpus of {CORPUS_UTTS * world} utterances dealt to {world} rank(s) by length bucket (parallel.shard_by_length), no collective",
           "l2": "inputs (2.1 GB/step) larger than L2, no flush needed"}
    if note:
        cfg["note"] = note
    return cfg


# --------------------------------------------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------------------------------------------
def run_b200(args):
    global N_FFT, HOP, FLOP_PER_FRAME, BYTES_PER_FRAME
    if args.n_fft != N_FFT:
        N_FFT = args.n_fft
        HOP = 200 if N_FFT == 400 else 160
        FLOP_PER_FRAME = {400: 20931 - 2 * 128 * 40 - 128, 1600: 49868}.get(N_FFT, FLOP_PER_FRAME)
        BYTES_PER_FRAME = 4 * HOP + 4 * N_MELS
    import torch.distributed as dist
    from speech_emotion_privacy_trust_b200 import _lib, extraction

    rank, local, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.lib().sept_init(N_MELS))

    from speech_emotion_privacy_trust_b200 import parallel
    placement = parallel.bind_host_to_gpu(local)                  # before any pinned allocation (host-buffer path)
    all_lengths = corpus_lengths(args.utts * world, 1234)        # ONE corpus for the whole job ...
    shards = parallel.shard_by_length(all_lengths, world)        # ... length-bucketed (0.5 s) and balanced over the ranks
    lengths = all_lengths[shards[rank]]
    shard_audio = np.array([all_lengths[sh].sum() for sh in shards], dtype=np.float64)
    if args.round_lengths > 1:                                    # debug only: every utterance starts on an aligned sample
        lengths = (lengths // args.round_lengths) * args.round_lengths
    utt_off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    wav = synth_corpus_device(lengths, 4321 + rank, dev)
    batch = extraction.RaggedAudio(wav, utt_off)
    lay = batch.layout(N_FFT, HOP)
    frames = lay.total_frames
    hours = float(lengths.sum()) / 16000 / 3600
    out = torch.empty((frames, N_MELS), dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput ("value") -------------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        extraction.logmel(batch, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out=out)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        time.sleep(0.3)
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    t0 = time.perf_counter()
    torch.cuda.nvtx.range_push("timed")                       # ncu --nvtx --nvtx-include "timed/" lists exactly these launches
    evs[0].record()
    for k in range(args.steps):
        extraction.logmel(batch, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out=out)
        evs[k + 1].record()
    barrier()
    torch.cuda.nvtx.range_pop()
    t1 = time.perf_counter()
    total_ms = evs[0].elapsed_time(evs[-1])
    kernel_ms = [evs[k].elapsed_time(evs[k + 1]) for k in range(args.steps)]     # one launch per step on this stream
    clocks = sampler.window(t0, t1) if sampler else None
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), out, lay, rank, world)

    # ---- end to end through the public API with HOST buffers ("e2e") ----------------------------------------
    if args.no_extras:
        e2e_ms = 0.0
    else:
        e2e_ms = measure_e2e(args, extraction, wav, utt_off, frames, out, dev, barrier)
    # ---- max over ranks --------------------------------------------------------------------------------------
    stats = torch.tensor([total_ms, e2e_ms, hours, float(frames)], dtype=torch.float64, device=dev)
    rank_ms = [total_ms / args.steps]
    if world > 1:
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = stats.clone()
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        every = [torch.empty_like(stats) for _ in range(world)]
        dist.all_gather(every, stats)
        rank_ms = [float(t[0]) / args.steps for t in every]
        total_ms, e2e_ms = float(mx[0]), float(mx[1])
        hours_all, frames_all = float(sm[2]), float(sm[3])
    else:
        hours_all, frames_all = hours, float(frames)
    sharding = {"policy": "parallel.shard_by_length: one corpus, 0.5 s length buckets, longest-first greedy balance",
                "utterances_total": int(args.utts * world), "audio_hours_per_rank_max_over_mean": float(shard_audio.max() / shard_audio.mean()),
                "rank_ms_per_step_max": max(rank_ms), "rank_ms_per_step_mean": sum(rank_ms) / len(rank_ms), "host_placement": placement}

    extras = {}
    if args.no_extras:
        extras = {"skipped": True}
    elif rank == 0 or world > 1:
        try:
            extras = secondary_metrics(args, dev, rank, world, batch if rank == 0 else None, hours)
        except Exception as exc:                                   # the headline number must not depend on the extras
            extras = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        peaks, peak_src = measured_peaks()
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        fp32_peak = sms * FP32_LANES_PER_SM * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6 / 1e12
        k_ms = statistics.mean(kernel_ms)
        ach_tf = FLOP_PER_FRAME * frames / (k_ms * 1e-3) / 1e12
        ach_gbs = BYTES_PER_FRAME * frames / (k_ms * 1e-3) / 1e9
        line = {
            "metric": "log-mel audio-hours/sec", "value": hours_all * args.steps / (total_ms * 1e-3), "unit": "audio-hours/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(world),
            "sharding": sharding,
            "clocks": clocks,
            "e2e": None if args.no_extras else {"value": hours_all / (e2e_ms * 1e-3), "unit": "audio-hours/s", "h2d_bytes_per_step": int(wav.numel() * 4),
                    "d2h_bytes_per_step": int(frames * N_MELS * 4), "ms_per_step": e2e_ms,
                    "api": "extraction.logmel_host(pinned host wav, utt_off) -> pinned host (frames,128)",
                    "pcm16_input": None if E2E_PCM16_MS is None else {
                        "ms_per_step_this_rank": E2E_PCM16_MS, "audio_hours_per_s_this_rank": hours / (E2E_PCM16_MS * 1e-3),
                        "h2d_bytes_per_step": int(wav.numel() * 2),
                        "note": "same call with 16-bit PCM host input (x/32768 on the device, as torchaudio.load does on the host)"}},
            "gpu_launches": args.steps,
            "roofline": {"bound": "fp32", "achieved": ach_tf, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach_tf / fp32_peak,
                         "traffic": profiled_traffic(frames), "traffic_source": "ncu --set full capture under profiles/ (dram__bytes_read+write of one launch, scaled by frames); not measured in this run",
                         "algorithmic_bytes": BYTES_PER_FRAME * frames, "kernel": "extract_kernel<16, frame-major>", "kernel_ms": k_ms,
                         "algorithmic_flop_per_frame": FLOP_PER_FRAME, "frames_per_launch": frames,
                         "peak_source": f"{sms} SMs x 128 FP32 lanes x 2 x sm_max_mhz of MEASURED_PEAKS.json ({peak_src}); "
                                        "the path is FP32-CUDA-core bound, not HBM or tensor bound (SURVEY 8d)",
                         "hbm": {"achieved": ach_gbs, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                                 "frac": ach_gbs / peaks.get("hbm_gbs", 6650.0), "algorithmic_bytes_per_frame": BYTES_PER_FRAME}},
            "extras": extras,
        }
        line["cpu_baseline"] = cpu_baseline() if (world == 1 and not args.no_extras) else None
        print(json.dumps(line))
    if sampler:
        sampler.stop()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(dst: Path, feats: torch.Tensor, lay, rank: int, world: int):
    """What the last timed extraction.logmel call returned, for comparing two builds output by output: DUMP_ROWS //
    world feature rows of this rank drawn with a seed fixed per rank (logmel.npy, float32), their row indices
    (logmel_rows.npy) and the per-utterance frame offsets of the layout (frame_offsets.npy), both float64.  With
    N > 1 every rank adds a _rank<r> suffix.  The total is about 34 MB at any N: 32 MiB of features, 0.5 MiB of
    row indices and 44 KB of frame offsets per rank."""
    dst.mkdir(parents=True, exist_ok=True)
    n = feats.shape[0]
    rows = np.sort(np.random.default_rng(rank).choice(n, size=min(DUMP_ROWS // world, n), replace=False))
    suffix = "" if world == 1 else f"_rank{rank}"
    np.save(dst / f"logmel{suffix}.npy", feats[torch.from_numpy(rows).to(feats.device)].cpu().numpy())
    np.save(dst / f"logmel_rows{suffix}.npy", rows.astype(np.float64))
    np.save(dst / f"frame_offsets{suffix}.npy", lay.frame_off_host.astype(np.float64))


def measure_e2e(args, extraction, wav, utt_off, frames, out, dev, barrier):
    host_wav = torch.empty(wav.numel(), dtype=torch.float32, pin_memory=True)
    host_wav.copy_(wav)
    host_out = torch.empty((frames, N_MELS), dtype=torch.float32, pin_memory=True)
    e2e_steps = max(2, min(args.steps, 5))
    extraction.logmel_host(host_wav, utt_off, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out_host=host_out, device=dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(e2e_steps):
        extraction.logmel_host(host_wav, utt_off, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out_host=host_out, device=dev)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1) / e2e_steps
    if not torch.equal(host_out[:1000], out[:1000].cpu()):
        raise SystemExit("bench.py: end-to-end result differs from the device-resident result")
    # the same pipeline fed with 16-bit PCM (what the corpora are on disk): half the host->device bytes
    global E2E_PCM16_MS
    pcm = torch.empty(wav.numel(), dtype=torch.int16, pin_memory=True)
    pcm.copy_((wav * 32767.0).round().to(torch.int16))
    extraction.logmel_host(pcm, utt_off, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out_host=host_out, device=dev)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for _ in range(e2e_steps):
        extraction.logmel_host(pcm, utt_off, n_fft=N_FFT, n_mels=N_MELS, hop=HOP, out_host=host_out, device=dev)
    p1.record()
    barrier()
    E2E_PCM16_MS = p0.elapsed_time(p1) / e2e_steps

    return e2e_ms


def cpu_baseline():
    threads = os.cpu_count() or 1
    n_sample = 600
    waves = cpu_sample_waves(n_sample, 1234)
    hours = sum(a.shape[1] for a in waves) / 16000 / 3600
    time_cpu_reference(waves[:50], threads)
    best = min(time_cpu_reference(waves, threads) for _ in range(2))
    return {"value": hours / best, "unit": "audio-hours/s", "cores": threads, "kind": "port",
            "sample": f"first {n_sample} utterances ({hours:.2f} audio-h) of the seed-1234 corpus, reference loop "
                      "(one utterance per call, transforms built per call), best of 2"}


def secondary_metrics(args, dev, rank, world, batch=None, hours=None):
    """BASELINE.json's second figure: cloak+GRL training utterances/sec (config 3), data parallel, B=32 per GPU; plus the
    other features the reference's extraction script computes per utterance (this rank's numbers, device resident)."""
    from benchmarks_train import cloak_kernel_bandwidth, eval_throughput, train_throughput
    out = train_throughput(dev, rank, world, steps=20, warmup=5)
    if world > 1 and os.environ.get("SEPT_BENCH_TRAIN_AB") == "1":           # A/B of the gradient exchange in one run
        ab = train_throughput(dev, rank, world, steps=20, warmup=5, overlap=True)
        out["two_bucket_overlap_ab"] = {k: ab[k] for k in ("value", "ms_per_step", "allreduce")}
    if rank == 0:
        out["cloak_eval"] = eval_throughput(dev)
        out["cloak_kernels"] = cloak_kernel_bandwidth(dev)
        if world == 1:
            from benchmarks_train import eval_cpu_baseline, train_cpu_baseline
            out["train_cpu_baseline"] = train_cpu_baseline()
            out["cloak_eval_cpu_baseline"] = eval_cpu_baseline()
    if batch is not None:
        out["other_features_this_rank"] = other_features(batch, hours, dev)
    if world > 1:
        out["speaker_stats_nccl_check"] = speaker_stats_nccl_check(dev, rank, world)
    if not args.no_bulk:
        bulk = bulk_extraction(dev, rank, world, args.bulk_hours)
        if rank == 0:
            out["bulk_extraction"] = bulk
    return out


def speaker_stats_nccl_check(dev, rank, world, n_utts=64, n_spk=10, seed=99):
    """SURVEY 8e row 2 on hardware: per-speaker statistics when every speaker's utterances are spread over the ranks
    (one NCCL all-gather of the partials + Chan merge) equal the statistics one rank computes over all utterances."""
    import torch.distributed as dist
    from speech_emotion_privacy_trust_b200 import normalization as nz, parallel
    from speech_emotion_privacy_trust_b200.extraction import Layout
    rng = np.random.default_rng(seed)                              # the same data on every rank
    frames = rng.integers(201, 1002, size=n_utts)
    spk = [f"s{int(rng.integers(n_spk))}" for _ in range(n_utts)]
    feats = [(rng.standard_normal((int(T), 128)) * 8 - 40).astype(np.float32) for T in frames]
    speakers = sorted(set(spk))

    def stats_of(idx, distributed):
        fo = np.concatenate([[0], np.cumsum([frames[i] for i in idx])]).astype(np.int64)
        lay = Layout(fo, torch.from_numpy(fo).to(dev), torch.zeros(len(fo), dtype=torch.int32, device=dev))
        feat = torch.from_numpy(np.concatenate([feats[i] for i in idx])).to(dev)
        who = [spk[i] for i in idx]
        return nz.speaker_stats_distributed(feat, lay, who, speakers) if distributed else nz.speaker_stats(feat, lay, who)
    mine = [int(i) for i in parallel.shard_by_length(frames * 160, world)[rank]]
    got = stats_of(mine, True).as_dict()
    want = stats_of(list(range(n_utts)), False).as_dict()
    worst = 0.0
    for s_ in speakers:
        for k in ("count", "mean", "std", "min", "max"):
            worst = max(worst, float(np.max(np.abs(got[s_][k] - want[s_][k]))))
    t = torch.tensor([worst], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t)
    if worst > 1e-3:
        raise SystemExit(f"bench.py: distributed speaker statistics differ from the single-rank ones by {worst}")
    return {"speakers": len(speakers), "utterances": n_utts, "max_abs_diff_vs_single_rank": worst, "collective": "all_gather of (count, mean, M2, min, max) partials"}


def bulk_extraction(dev, rank, world, total_hours=1000.0, chunk_utts=CORPUS_UTTS):
    """BASELINE.json configs[3]: bulk log-mel extraction of `total_hours` synthetic audio-hours (600 000 utterances of
    2-10 s for 1000 h), length-bucketed and sharded over the ranks by parallel.shard_by_length.  1000 h of fp32 waveform
    (230 GB) exceed one GPU, so every rank synthesises its shard on the device in corpus-sized chunks (2.1 GB), extracts
    the chunk (one launch, timed with CUDA events) and drops it; the figure is total audio-hours over the slowest rank's
    summed kernel time -- strong scaling of a fixed job, inputs resident in HBM."""
    import torch.distributed as dist
    from speech_emotion_privacy_trust_b200 import extraction, parallel
    n_utts = int(round(total_hours * 600))                         # mean 6 s
    lengths = corpus_lengths(n_utts, 4321)
    t0 = time.perf_counter()
    mine = lengths[parallel.shard_by_length(lengths, world)[rank]]
    t_shard = time.perf_counter() - t0
    out = None
    ms, frames, n_launch = 0.0, 0, 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for c, a in enumerate(range(0, len(mine), chunk_utts)):
        lens = mine[a:a + chunk_utts]
        off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        batch = extraction.RaggedAudio(synth_corpus_device(lens, 777 + 1000 * rank + c, dev), off)
        lay = batch.layout(800, 160)
        if out is None or out.shape[0] < lay.total_frames:
            out = torch.empty((int(lay.total_frames * 1.05), N_MELS), dtype=torch.float32, device=dev)
        if c == 0:
            extraction.logmel(batch, n_fft=800, n_mels=N_MELS, hop=160, out=out[:lay.total_frames])     # warm
        e0.record()
        extraction.logmel(batch, n_fft=800, n_mels=N_MELS, hop=160, out=out[:lay.total_frames])
        e1.record()
        torch.cuda.synchronize(dev)
        ms += e0.elapsed_time(e1)
        frames += lay.total_frames
        n_launch += 1
        del batch
    t = torch.tensor([ms, float(mine.sum()) / 16000 / 3600, float(frames)], dtype=torch.float64, device=dev)
    mx, sm = t.clone(), t.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    hours = float(sm[1])
    return {"workload": f"{hours:.0f} audio-hours, {n_utts} utterances of 2-10 s, length-bucketed over {world} rank(s), chunks of {chunk_utts} utterances synthesised on the device",
            "audio_hours": hours, "kernel_ms_slowest_rank": float(mx[0]), "kernel_ms_mean_rank": float(sm[0]) / world,
            "audio_hours_per_s": hours / (float(mx[0]) * 1e-3), "launches_this_rank": n_launch, "frames_total": float(sm[2]),
            "host_sharding_s": t_shard, "scaling": "strong"}


def other_features(batch, hours, dev, steps=5):
    """audio-hours/s of log-mel n_fft=1600 (mel2), MFCC-40 x3 streams, and all three features of
    audio_feature_extraction.py:185-187 back to back, with their FP32 roofline fractions (BASELINE.md section 3)."""
    from speech_emotion_privacy_trust_b200 import extraction
    peaks, _ = measured_peaks()
    fp32_peak = torch.cuda.get_device_properties(dev).multi_processor_count * FP32_LANES_PER_SM * 2 * peaks.get("sm_max_mhz", 1965.0) * 1e6

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / steps

    f800 = batch.layout(800, 160).total_frames
    f400 = batch.layout(400, 200).total_frames
    mel_out = torch.empty((f800, N_MELS), dtype=torch.float32, device=dev)
    mfcc_out = torch.empty(f400 * 120, dtype=torch.float32, device=dev)
    res = {}
    ms = timed(lambda: extraction.logmel(batch, n_fft=1600, n_mels=N_MELS, hop=160, out=mel_out))
    res["logmel_1600"] = {"audio_hours_per_s": hours / (ms * 1e-3), "ms": ms, "fp32_frac": 49868 * f800 / (ms * 1e-3) / fp32_peak}
    ms = timed(lambda: extraction.mfcc(batch, out=mfcc_out))
    res["mfcc_3streams"] = {"audio_hours_per_s": hours / (ms * 1e-3), "ms": ms, "fp32_frac": 3 * 20931 * f400 / (ms * 1e-3) / fp32_peak}

    def all_three():
        extraction.logmel(batch, n_fft=800, n_mels=N_MELS, hop=160, out=mel_out)
        extraction.logmel(batch, n_fft=1600, n_mels=N_MELS, hop=160, out=mel_out)
        extraction.mfcc(batch, out=mfcc_out)
    ms = timed(all_three)
    flop = (22999 + 49868) * f800 + 3 * 20931 * f400
    res["all_three"] = {"audio_hours_per_s": hours / (ms * 1e-3), "ms": ms, "fp32_frac": flop / (ms * 1e-3) / fp32_peak}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary metric, e2e and cpu_baseline (profiling runs)")
    ap.add_argument("--n-fft", type=int, default=N_FFT, help="debug only: time another FFT size (the metric is quoted on 800)")
    ap.add_argument("--round-lengths", type=int, default=1, help="debug only: round utterance lengths down to a multiple (alignment experiments)")
    ap.add_argument("--utts", type=int, default=CORPUS_UTTS, help="utterances per GPU (debug only; the metric is quoted on the default)")
    ap.add_argument("--no-bulk", action="store_true", help="skip the 1000-audio-hour bulk extraction (BASELINE.json configs[3]) in extras")
    ap.add_argument("--bulk-hours", type=float, default=1000.0, help="size of the bulk extraction job in extras")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a seeded sample of the last step's "
                                                          "log-mel features and its frame offsets to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computes; the reference arm keeps no outputs")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
