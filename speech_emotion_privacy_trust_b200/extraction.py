"""Batched B200 feature extraction: the new ragged-batch entry points above the C ABI.

The reference extracts one utterance per Python call on the CPU (feature_extraction/audio_feature_extraction.py:
180-189).  Here a whole batch of utterances is one ragged device buffer and one kernel launch per feature.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from . import _lib

SAMPLE_RATE = 16000
HOP_MEL = 160            # audio_feature_extraction.py:32
N_FFT_MFCC, HOP_MFCC, N_MFCC = 400, 200, 40   # torchaudio MFCC defaults used by audio_feature_extraction.py:17


@dataclass
class Layout:
    """Frame / work-item offsets of a ragged batch for one (n_fft, hop)."""
    frame_off_host: np.ndarray       # int64 [n+1]
    frame_off: torch.Tensor          # device int64 [n+1]
    item_off: torch.Tensor           # device int32 [n+1]
    n_items: int = 0                 # item_off[n]: work items of the batch (0 with the all-zero item_off of frame layouts)

    @property
    def total_frames(self) -> int:
        return int(self.frame_off_host[-1])

    def frames(self, u: int) -> int:
        return int(self.frame_off_host[u + 1] - self.frame_off_host[u])


class RaggedAudio:
    """Utterances back to back in one device buffer: wav[utt_off[u]:utt_off[u+1]] (16 kHz mono fp32)."""

    def __init__(self, wav: torch.Tensor, utt_off_host: np.ndarray):
        _lib.require_cuda(wav)
        if wav.dtype != torch.float32 or wav.dim() != 1 or not wav.is_contiguous():
            raise ValueError("wav must be a contiguous 1-D float32 tensor")
        self.wav = wav
        self.utt_off_host = np.ascontiguousarray(utt_off_host, dtype=np.int64)
        if self.utt_off_host.ndim != 1 or len(self.utt_off_host) < 1 or self.utt_off_host[-1] > wav.numel():
            raise ValueError("utt_off must be a 1-D offset array within wav")
        self.utt_off = torch.from_numpy(self.utt_off_host).to(wav.device, non_blocking=True)
        self._layouts: dict[tuple[int, int], Layout] = {}

    @classmethod
    def from_list(cls, waves: Sequence, device="cuda") -> "RaggedAudio":
        arrs = [np.asarray(w.detach().cpu() if torch.is_tensor(w) else w, dtype=np.float32).reshape(-1) for w in waves]
        off = np.zeros(len(arrs) + 1, dtype=np.int64)
        np.cumsum([len(a) for a in arrs], out=off[1:])
        host = torch.from_numpy(np.concatenate(arrs) if arrs else np.zeros(0, np.float32))
        return cls(host.to(device), off)

    @property
    def n_utts(self) -> int:
        return len(self.utt_off_host) - 1

    def layout(self, n_fft: int, hop: int) -> Layout:
        key = (n_fft, hop)
        if key not in self._layouts:
            n = self.n_utts
            frame_off = np.zeros(n + 1, dtype=np.int64)
            item_off = np.zeros(n + 1, dtype=np.int32)
            _lib.check(_lib.lib().sept_extract_layout(self.utt_off_host.ctypes.data, n, n_fft, hop,
                                                      frame_off.ctypes.data, item_off.ctypes.data))
            dev = self.wav.device
            self._layouts[key] = Layout(frame_off, torch.from_numpy(frame_off).to(dev), torch.from_numpy(item_off).to(dev),
                                        int(item_off[-1]))
        return self._layouts[key]


def resample(batch: "RaggedAudio", orig_freq: int, new_freq: int = SAMPLE_RATE) -> "RaggedAudio":
    """Band-limited sinc resampling of every utterance (torchaudio.transforms.Resample(orig_freq, new_freq) as the
    reference applies it to 44.1 kHz corpora, audio_feature_extraction.py:139-141); returns a new ragged batch."""
    if orig_freq == new_freq:
        return batch
    n = batch.n_utts
    out_off = np.zeros(n + 1, dtype=np.int64)
    _lib.check(_lib.lib().sept_resample_layout(batch.utt_off_host.ctypes.data, n, orig_freq, new_freq, out_off.ctypes.data))
    dev = batch.wav.device
    out = torch.empty(int(out_off[-1]), dtype=torch.float32, device=dev)
    d_out_off = torch.from_numpy(out_off).to(dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sept_resample_f32(batch.wav.data_ptr(), batch.utt_off.data_ptr(), d_out_off.data_ptr(), n,
                                                int(out_off[-1]), orig_freq, new_freq, out.data_ptr(),
                                                torch.cuda.current_stream(dev).cuda_stream))
    res = RaggedAudio.__new__(RaggedAudio)
    res.wav, res.utt_off_host, res.utt_off, res._layouts = out, out_off, d_out_off, {}
    return res


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def logmel(batch: RaggedAudio, n_fft: int = 800, n_mels: int = 128, hop: int = HOP_MEL, band_major: bool = False,
           deriv: bool = False, out: torch.Tensor | None = None) -> tuple[torch.Tensor, Layout]:
    """log-mel dB of every utterance of the batch (the arithmetic of mel_spectrogram(), reference :29-46).

    Returns (features, layout).  Frame-major (default): features is (total_frames, n_mels) and utterance u is rows
    layout.frame_off[u]:layout.frame_off[u+1] -- the (T, 128) matrix preprocess_adversary_data.py:345 builds with
    mel1[0].T.  band_major: flat buffer whose utterance u is an (n_mels, T_u) block at frame_off[u] * n_mels.
    """
    lay = batch.layout(n_fft, hop)
    dev = batch.wav.device
    if out is None:
        shape = (lay.total_frames * n_mels,) if band_major else (lay.total_frames, n_mels)
        out = torch.empty(shape, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sept_logmel_f32(batch.wav.data_ptr(), batch.utt_off.data_ptr(), lay.frame_off.data_ptr(),
                                              lay.item_off.data_ptr(), batch.n_utts, n_fft, hop, n_mels, int(deriv),
                                              1 if band_major else 0, out.data_ptr(), _stream(dev)))
    return out, lay


class LogMelFunction(torch.autograd.Function):
    """Frame-major log-mel dB with a waveform gradient: forward is one sept_logmel_f32 launch, backward one
    sept_logmel_bwd_f32 launch (recomputes the spectrum from the saved waveform; no double backward)."""

    @staticmethod
    def forward(ctx, wav, batch, n_fft, n_mels, hop):
        out, lay = logmel(batch, n_fft, n_mels, hop)
        ctx.save_for_backward(wav)
        ctx.batch, ctx.lay, ctx.shape = batch, lay, (n_fft, n_mels, hop)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        (wav,) = ctx.saved_tensors
        batch, lay = ctx.batch, ctx.lay
        n_fft, n_mels, hop = ctx.shape
        lib = _lib.lib()
        dwav = torch.zeros_like(wav)                              # samples outside every utterance get no gradient
        ws = torch.empty(max(1, lib.sept_logmel_bwd_workspace_bytes(n_fft, hop, lay.n_items)), dtype=torch.uint8,
                         device=wav.device)
        grad = grad.contiguous()
        with torch.cuda.device(wav.device):
            _lib.check(lib.sept_logmel_bwd_f32(wav.data_ptr(), batch.utt_off.data_ptr(), lay.frame_off.data_ptr(),
                                               lay.item_off.data_ptr(), batch.n_utts, lay.n_items, n_fft, hop, n_mels,
                                               grad.data_ptr(), ws.data_ptr(), dwav.data_ptr(), _stream(wav.device)))
        return dwav, None, None, None, None


def logmel_grad(batch: RaggedAudio, n_fft: int = 800, n_mels: int = 128, hop: int = HOP_MEL, band_major: bool = False,
                deriv: bool = False) -> tuple[torch.Tensor, Layout]:
    """logmel() with a gradient: the (total_frames, n_mels) frame-major features carry a grad_fn back to batch.wav.

    Values are bit-identical to logmel().  The backward writes d/d wav for every sample of every utterance (zero
    elsewhere), deterministically.  Only the frame-major waveform stream is differentiable: band_major (one transpose in
    torch away) and deriv raise ValueError."""
    if band_major:
        raise ValueError("logmel_grad: only the frame-major layout has a gradient; transpose the result instead")
    if deriv:
        raise ValueError("logmel_grad: the np.gradient stream (deriv) has no gradient")
    lay = batch.layout(n_fft, hop)
    return LogMelFunction.apply(batch.wav, batch, n_fft, n_mels, hop), lay


def mfcc(batch: RaggedAudio, out: torch.Tensor | None = None) -> tuple[torch.Tensor, Layout]:
    """MFCC-40 of x, np.gradient(x) and np.gradient(x, 2) (the arithmetic of mfcc(), reference :15-26).

    Returns (flat, layout): utterance u is the (120, T_u) block flat[frame_off[u]*120 : frame_off[u+1]*120]."""
    lay = batch.layout(N_FFT_MFCC, HOP_MFCC)
    dev = batch.wav.device
    tf = lay.total_frames
    if out is None:
        out = torch.empty(tf * 3 * N_MFCC, dtype=torch.float32, device=dev)
    scratch = torch.empty(tf * 257, dtype=torch.float32, device=dev)
    utt_max = torch.empty(2 * batch.n_utts, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().sept_mfcc_f32(batch.wav.data_ptr(), batch.utt_off.data_ptr(), lay.frame_off.data_ptr(),
                                            lay.item_off.data_ptr(), batch.n_utts, tf, scratch.data_ptr(),
                                            utt_max.data_ptr(), out.data_ptr(), _stream(dev)))
    return out, lay


class MfccFunction(torch.autograd.Function):
    """MFCC blocks with a waveform gradient: forward is one sept_mfcc_f32 call, backward one sept_mfcc_bwd_f32 call
    (recomputes the mel power from the saved waveform; no double backward)."""

    @staticmethod
    def forward(ctx, wav, batch):
        out, lay = mfcc(batch)
        ctx.save_for_backward(wav)
        ctx.batch, ctx.lay = batch, lay
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        (wav,) = ctx.saved_tensors
        batch, lay = ctx.batch, ctx.lay
        lib = _lib.lib()
        dwav = torch.zeros_like(wav)                              # samples outside every utterance get no gradient
        ws = torch.empty(max(1, lib.sept_mfcc_bwd_workspace_bytes(batch.n_utts, lay.total_frames, lay.n_items)),
                         dtype=torch.uint8, device=wav.device)
        grad = grad.contiguous()
        with torch.cuda.device(wav.device):
            _lib.check(lib.sept_mfcc_bwd_f32(wav.data_ptr(), batch.utt_off.data_ptr(), lay.frame_off.data_ptr(),
                                             lay.item_off.data_ptr(), batch.n_utts, lay.total_frames, lay.n_items,
                                             grad.data_ptr(), ws.data_ptr(), dwav.data_ptr(), _stream(wav.device)))
        return dwav, None


def mfcc_grad(batch: RaggedAudio) -> tuple[torch.Tensor, Layout]:
    """mfcc() with a gradient: the flat (120, T_u) blocks carry a grad_fn back to batch.wav.

    Values are bit-identical to mfcc().  The backward is what torch autograd gives through the reference's chain (the
    top_db floor sends the gradient of floored values to the utterance's maximum) and writes d/d wav for every sample
    of every utterance (zero elsewhere), deterministically."""
    lay = batch.layout(N_FFT_MFCC, HOP_MFCC)
    return MfccFunction.apply(batch.wav, batch), lay


def split_band_major(flat: torch.Tensor, lay: Layout, rows: int) -> list[torch.Tensor]:
    """Views (rows, T_u) of a band-major flat buffer, one per utterance."""
    fo = lay.frame_off_host
    return [flat[fo[u] * rows:fo[u + 1] * rows].view(rows, -1) for u in range(len(fo) - 1)]


# ---- host-buffer entry point: copies pipelined against the kernel ----------------------------------------------
def logmel_host(wav_host: torch.Tensor, utt_off_host: np.ndarray, n_fft: int = 800, n_mels: int = 128, hop: int = HOP_MEL,
                out_host: torch.Tensor | None = None, device="cuda", chunk_samples: int = 1 << 24, n_streams: int = 3,
                sync: bool = True):
    """log-mel dB for a ragged batch that lives in HOST memory, result back in host memory (frame-major).

    wav_host may also be 16-bit PCM (int16): it is converted on the device as x / 32768, exactly what torchaudio.load does
    on the host before the reference's callables see the audio, and halves the host->device bytes.
    The batch is cut into chunks of about `chunk_samples` samples at utterance boundaries; each chunk is copied to the
    device, extracted and copied back on one of `n_streams` streams, so the H2D copy, the kernel and the D2H copy of
    neighbouring chunks overlap (PCIe is full duplex).  Pass pinned tensors to get asynchronous copies.
    Returns (out_host, frame_off_host).  With sync=True (default) the call returns once the last device->host copy has
    landed, so out_host can be read straight away; sync=False returns as soon as the work is queued (the caller's current
    stream is ordered after it: synchronise that stream, or the device, before touching out_host)."""
    dev = torch.device(device)
    if wav_host.is_cuda or wav_host.dtype not in (torch.float32, torch.int16) or wav_host.dim() != 1:
        raise ValueError("wav_host must be a 1-D float32 (or 16-bit PCM int16) host tensor")
    pcm16 = wav_host.dtype == torch.int16
    lib = _lib.lib()
    off = np.ascontiguousarray(utt_off_host, dtype=np.int64)
    n = len(off) - 1
    frame_off = np.zeros(n + 1, dtype=np.int64)
    item_off = np.zeros(n + 1, dtype=np.int32)
    _lib.check(lib.sept_extract_layout(off.ctypes.data, n, n_fft, hop, frame_off.ctypes.data, item_off.ctypes.data))
    total_frames = int(frame_off[-1])
    if out_host is None:
        out_host = torch.empty((total_frames, n_mels), dtype=torch.float32, pin_memory=True)
    # chunk boundaries at utterance starts
    bounds = [0]
    while bounds[-1] < n:
        a = bounds[-1]
        b = int(np.searchsorted(off, off[a] + chunk_samples, side="right")) - 1
        bounds.append(min(n, max(b, a + 1)))
    n_chunks = len(bounds) - 1
    # all per-chunk offset tables in one pinned buffer, one H2D copy
    per = [(bounds[c], bounds[c + 1]) for c in range(n_chunks)]
    words = sum(3 * (b - a + 1) for a, b in per)
    tab_host = torch.empty(words, dtype=torch.int64, pin_memory=True)   # torch's pinned allocator is stream aware: the
                                                                        # block is not reused before the copy below has run
    pos, slots = 0, []
    for a, b in per:
        k = b - a + 1
        tab_host[pos:pos + k] = torch.from_numpy(off[a:b + 1] - off[a])
        tab_host[pos + k:pos + 2 * k] = torch.from_numpy(frame_off[a:b + 1] - frame_off[a])
        tab_host[pos + 2 * k:pos + 3 * k].view(torch.int32)[:k] = torch.from_numpy(item_off[a:b + 1] - item_off[a])
        slots.append((pos, k))
        pos += 3 * k
    with torch.cuda.device(dev):
        main = torch.cuda.current_stream(dev)
        tab_dev = tab_host.to(dev, non_blocking=True)
        max_samples = max(int(off[b] - off[a]) for a, b in per)
        max_frames = max(int(frame_off[b] - frame_off[a]) for a, b in per)
        streams = [torch.cuda.Stream(dev) for _ in range(min(n_streams, n_chunks))]
        bufs = [(torch.empty(max_samples, dtype=torch.float32, device=dev),
                 torch.empty((max_frames, n_mels), dtype=torch.float32, device=dev)) for _ in streams]
        pcm_bufs = [torch.empty(max_samples, dtype=torch.int16, device=dev) for _ in streams] if pcm16 else None
        ready = torch.cuda.Event()
        ready.record(main)
        for c, (a, b) in enumerate(per):
            s = streams[c % len(streams)]
            wbuf, obuf = bufs[c % len(streams)]
            ns, nf = int(off[b] - off[a]), int(frame_off[b] - frame_off[a])
            p, k = slots[c]
            with torch.cuda.stream(s):
                if c < len(streams):
                    s.wait_event(ready)
                if pcm16:
                    pbuf = pcm_bufs[c % len(streams)]
                    pbuf[:ns].copy_(wav_host[int(off[a]):int(off[b])], non_blocking=True)
                    _lib.check(lib.sept_pcm16_to_f32(pbuf.data_ptr(), ns, wbuf.data_ptr(), s.cuda_stream))
                else:
                    wbuf[:ns].copy_(wav_host[int(off[a]):int(off[b])], non_blocking=True)
                base = tab_dev.data_ptr() + 8 * p
                _lib.check(lib.sept_logmel_f32(wbuf.data_ptr(), base, base + 8 * k, base + 16 * k, b - a, n_fft, hop, n_mels,
                                               0, 0, obuf.data_ptr(), s.cuda_stream))
                out_host[frame_off[a]:frame_off[b]].copy_(obuf[:nf], non_blocking=True)
        for s in streams:
            main.wait_stream(s)
        for wbuf, obuf in bufs:
            wbuf.record_stream(main)
            obuf.record_stream(main)
        for pbuf in pcm_bufs or []:
            pbuf.record_stream(main)
        if sync:
            done = torch.cuda.Event()
            done.record(main)
            done.synchronize()
    return out_host, frame_off
