"""Sinc resampler (the step before the hot path for 44.1 kHz corpora): oracle vs the golden vectors produced by
torchaudio.transforms.Resample -- the call the reference makes (audio_feature_extraction.py:139-141) --, the library's
row table vs the oracle kernel (CPU), and the CUDA kernel vs both (GPU)."""
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import restate

REPO = Path(__file__).resolve().parents[1]
GOLD = np.load(REPO / "tests" / "golden" / "resample.npz")
TOL = 5e-6          # absolute, signals peak-normalised to 0.3: fp32 accumulation over ~35 (here) or 475 (torchaudio) taps


def test_oracle_matches_torchaudio_golden():
    for i in range(4):
        y = restate.resample(GOLD[f"in{i}"], 44100, 16000)
        assert y.shape == GOLD[f"out{i}"].shape                      # torchaudio's cut (restate.resample_length)
        assert np.max(np.abs(y - GOLD[f"out{i}"])) < TOL
    assert np.max(np.abs(restate.resample(GOLD["in_48k"], 48000, 16000) - GOLD["out_48k"])) < TOL
    assert [len(restate.resample(np.zeros(n), 44100, 16000)) for n in (1, 441, 442, 44100)] == [1, 160, 161, 16000]


@pytest.mark.parametrize("orig,up,rates", [(441, 160, (44100, 16000)), (3, 1, (48000, 16000)), (1, 2, (8000, 16000)),
                                           (147, 160, (44100, 48000)), (160, 441, (16000, 44100))])
def test_library_row_table_matches_oracle_kernel(tmp_path, orig, up, rates):
    exe = tmp_path / "rows"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", str(REPO / "speech_emotion_privacy_trust_b200" / "csrc"),
                    str(REPO / "tests" / "hostsim" / "resample_rows.cpp"), "-o", str(exe)], check=True)
    subprocess.run([str(exe), str(orig), str(up), str(tmp_path / "rows.bin")], check=True)
    raw = np.fromfile(tmp_path / "rows.bin", np.int32)
    width, taps = int(raw[0]), int(raw[1])
    k_lo = raw[2:2 + up]
    rows = raw[2 + up:].view(np.float32).reshape(up, taps)
    kern, w_ref, o_ref, n_ref = restate.sinc_resample_kernel(*rates)
    assert (width, orig, up) == (w_ref, o_ref, n_ref)
    full = np.zeros_like(kern)
    kept = np.zeros(kern.shape, dtype=bool)
    for j in range(up):
        full[j, k_lo[j]:k_lo[j] + taps] = rows[j]
        kept[j, k_lo[j]:k_lo[j] + taps] = True
    assert np.max(np.abs(full - kern)[kept]) < 1e-7                   # float rounding of the kept taps
    assert np.max(np.abs(kern[~kept]), initial=0.0) < 1e-30           # what is cut off: cos^2(pi/2) residue of the window
    assert taps <= 2 * width + 4


@pytest.mark.gpu
def test_cuda_resampler_vs_golden_and_oracle():
    from speech_emotion_privacy_trust_b200 import extraction, synth
    waves = [GOLD[f"in{i}"] for i in range(4)]
    batch = extraction.RaggedAudio.from_list(waves)
    out = extraction.resample(batch, 44100, 16000)
    off = out.utt_off_host
    for i in range(4):
        got = out.wav[off[i]:off[i + 1]].cpu().numpy()
        assert got.shape == GOLD[f"out{i}"].shape
        assert np.max(np.abs(got - GOLD[f"out{i}"])) < TOL
        assert np.max(np.abs(got - restate.resample(waves[i], 44100, 16000))) < TOL
    b48 = extraction.RaggedAudio.from_list([GOLD["in_48k"]])
    assert np.max(np.abs(extraction.resample(b48, 48000, 16000).wav.cpu().numpy() - GOLD["out_48k"])) < TOL
    # MSP-Improv-shaped path: 44.1 kHz -> 16 kHz -> log-mel equals log-mel of the oracle's resampled audio
    rng = np.random.default_rng(12)
    w44 = [synth.speech_shaped(int(n), rng) for n in (44100, 61234, 30011)]
    r = extraction.resample(extraction.RaggedAudio.from_list(w44), 44100)
    mel, lay = extraction.logmel(r, n_fft=800)
    fo = lay.frame_off_host
    for u, w in enumerate(w44):
        ref = restate.mel_spectrogram(restate.resample(w, 44100, 16000)[None], 800, 128, dtype=np.float64)[0]
        got = mel[fo[u]:fo[u + 1]].cpu().numpy().T
        strong = ref > ref.max(axis=0, keepdims=True) - 50.0
        assert got.shape == ref.shape and np.max(np.abs(got - ref)[strong]) < 1e-3
    assert extraction.resample(r, 16000, 16000) is r
    # other rate pairs (other tile shapes of the tiled kernel; utterance boundaries inside a CTA's sample range)
    rng = np.random.default_rng(13)
    for f_in, f_out in ((44100, 48000), (16000, 44100), (8000, 16000), (22050, 16000)):
        ws = [(0.3 * rng.standard_normal(int(n))).astype(np.float32) for n in (977, 12001, 1, 3333, 40, 20011)]
        res = extraction.resample(extraction.RaggedAudio.from_list(ws), f_in, f_out)
        o = res.utt_off_host
        for u, w in enumerate(ws):
            ref = restate.resample(w, f_in, f_out)
            got = res.wav[o[u]:o[u + 1]].cpu().numpy()
            assert got.shape == ref.shape, (f_in, f_out, u)
            assert np.max(np.abs(got - ref)) < TOL, (f_in, f_out, u)


@pytest.mark.gpu
def test_cuda_simple_kernel_fallback_in_a_fresh_process():
    """Rate pairs whose tables do not fit shared memory take the one-thread-per-sample kernel; SEPT_RESAMPLE_SIMPLE=1 (read
    once per process) forces it, so the same golden comparison runs in a child process with the variable set."""
    import os
    import sys
    code = (
        "import numpy as np, sys\n"
        f"sys.path.insert(0, {str(REPO)!r})\n"
        "from speech_emotion_privacy_trust_b200 import extraction\n"
        f"g = np.load({str(REPO / 'tests' / 'golden' / 'resample.npz')!r})\n"
        "b = extraction.RaggedAudio.from_list([g[f'in{i}'] for i in range(4)])\n"
        "o = extraction.resample(b, 44100, 16000); off = o.utt_off_host\n"
        "err = max(float(np.max(np.abs(o.wav[off[i]:off[i+1]].cpu().numpy() - g[f'out{i}']))) for i in range(4))\n"
        "print('ERR', err)\n")
    env = dict(os.environ, SEPT_RESAMPLE_SIMPLE="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert float(r.stdout.split("ERR")[1]) < TOL
