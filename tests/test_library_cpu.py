"""CPU-only checks of the boundary: the C-ABI library builds/loads and exports every symbol include/sept.h declares,
host-side helpers behave, compute calls fail loudly without a GPU, and the kernel's index algebra (run lane by lane on
the host, tests/hostsim) reproduces the reference's golden vectors."""
import ctypes
import re
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"


def test_library_exports_every_declared_symbol():
    from speech_emotion_privacy_trust_b200 import _lib
    header = (REPO / "include" / "sept.h").read_text()
    declared = set(re.findall(r"\b(sept_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    handle = _lib.lib()
    for name in declared:
        assert getattr(handle, name) is not None
    assert handle.sept_version() >= 100
    assert [handle.sept_frames_per_item(n) for n in (400, 800, 1600, 1024)] == [8, 4, 2, 0]


def test_signatures_are_read_from_the_header():
    """The ctypes signatures come from include/sept.h: pointers and the stream as c_void_p, every scalar at its width (a
    c_int where the header says int64_t would truncate without an error)."""
    from speech_emotion_privacy_trust_b200 import _lib
    handle = _lib.lib()
    p, i, u64, f = ctypes.c_void_p, ctypes.c_int, ctypes.c_uint64, ctypes.c_float
    fn = handle.sept_cloak_fwd_f32
    assert fn.restype is i
    assert fn.argtypes == [p, p, p, p, p, u64, u64, p, i, f, f, f, i, i, p, p, p, p]
    fn = handle.sept_logmel_bwd_workspace_bytes
    assert fn.restype is ctypes.c_size_t and fn.argtypes == [i, i, ctypes.c_int64]
    fn = handle.sept_last_error
    assert fn.restype is ctypes.c_char_p and fn.argtypes == []


def test_signature_parser_rejects_an_unknown_type():
    from speech_emotion_privacy_trust_b200 import _lib
    good = "int sept_a(const double* x, /* int64_t in a comment */ int64_t n,\n           sept_stream_t s);"
    assert _lib.signatures(good) == {"sept_a": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p])}
    with pytest.raises(RuntimeError, match="'double'"):
        _lib.signatures("int sept_b(double x);")
    with pytest.raises(RuntimeError, match="'uint64_t'"):
        _lib.signatures("uint64_t sept_c(void);")


def test_loader_refuses_a_stale_library(tmp_path, monkeypatch):
    """VERDICT r1: a prebuilt .so compiled from other sources than the tree holds must never be tested silently.  The
    library carries the sha256 of its sources; the loader compares it with the tree and rebuilds or raises."""
    from speech_emotion_privacy_trust_b200 import _lib, build
    assert build.built_hash() == build.source_hash() and not build.stale()
    assert _lib.lib().sept_source_hash().decode() == "SEPT_SRC_HASH=" + build.source_hash()
    # a copy whose embedded hash is wrong + no compiler: loading must raise, not fall through
    fake = tmp_path / "libsept_b200.so"
    blob = build.LIB.read_bytes().replace(build.source_hash().encode(), b"0" * 64)
    fake.write_bytes(blob)
    monkeypatch.setattr(build, "LIB", fake)
    monkeypatch.setattr(build, "_nvcc", lambda: (_ for _ in ()).throw(RuntimeError("nvcc not found")))
    monkeypatch.setattr(_lib, "_LIB", None)
    assert build.stale()
    with pytest.raises(RuntimeError, match="stale"):
        _lib.lib()
    # the mtime of the sources plays no role (the tree is copied to the GPU box): touching a file is not "stale"
    monkeypatch.undo()
    src = CSRC / "philox.cuh"
    src.touch()
    assert not build.stale()


def test_layout_helper_matches_reference_frame_rule():
    from speech_emotion_privacy_trust_b200 import _lib
    lens = np.array([801, 1600, 4000, 7777, 16000, 48001], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    for n_fft, hop in ((800, 160), (1600, 160), (400, 200)):
        if n_fft == 1600:
            lens2, off2 = lens[2:], np.concatenate([[0], np.cumsum(lens[2:])]).astype(np.int64)
        else:
            lens2, off2 = lens, off
        fo = np.zeros(len(lens2) + 1, np.int64)
        io = np.zeros(len(lens2) + 1, np.int32)
        assert _lib.lib().sept_extract_layout(off2.ctypes.data, len(lens2), n_fft, hop, fo.ctypes.data, io.ctypes.data) == 0
        assert list(np.diff(fo)) == [1 + n // hop for n in lens2]          # T = 1 + N // hop (center=True)
        fpw = _lib.lib().sept_frames_per_item(n_fft)
        assert list(np.diff(io)) == [-(-(1 + n // hop) // fpw) for n in lens2]


def test_layout_helper_rejects_what_the_reference_rejects():
    from speech_emotion_privacy_trust_b200 import _lib
    off = np.array([0, 400], dtype=np.int64)                 # N == n_fft/2: torch.stft's reflect pad raises
    fo, io = np.zeros(2, np.int64), np.zeros(2, np.int32)
    rc = _lib.lib().sept_extract_layout(off.ctypes.data, 1, 800, 160, fo.ctypes.data, io.ctypes.data)
    assert rc == _lib.SEPT_E_TOO_SHORT
    with pytest.raises(RuntimeError, match="reflect padding"):
        _lib.check(rc)
    rc = _lib.lib().sept_extract_layout(off.ctypes.data, 1, 1024, 160, fo.ctypes.data, io.ctypes.data)
    assert rc == _lib.SEPT_E_UNSUPPORTED
    with pytest.raises(ValueError, match="n_fft=1024"):
        _lib.check(rc)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_compute_fails_loudly_without_a_gpu():
    from speech_emotion_privacy_trust_b200 import _lib, extraction
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        extraction.RaggedAudio(torch.zeros(1000), np.array([0, 1000]))
    buf = (ctypes.c_float * 16)()
    rc = _lib.lib().sept_grl_bwd_f32(ctypes.addressof(buf), 1.0, 16, ctypes.addressof(buf), None)
    assert rc == _lib.SEPT_E_CUDA


@pytest.fixture(scope="module")
def hostsim(tmp_path_factory):
    exe = tmp_path_factory.mktemp("hostsim") / "hostsim"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), str(REPO / "tests" / "hostsim" / "hostsim.cpp"), "-o", str(exe)],
                   check=True)
    return exe


@pytest.mark.parametrize("i", [0, 2, 3])
@pytest.mark.parametrize("key,n_fft,hop", [("mel1", 800, 160), ("mel2", 1600, 160), (None, 400, 200)])
def test_kernel_phase_functions_on_host(hostsim, golden_extraction, tmp_path, i, key, n_fft, hop):
    """The per-lane phase functions the CUDA kernel runs (csrc/extract_core.cuh), executed lane by lane on the CPU,
    against the reference's golden log-mel (n_fft 800/1600) or the fp64 oracle (n_fft 400)."""
    from oracle import restate
    wav = golden_extraction[f"wav{i}"]
    wav.tofile(tmp_path / "w.f32")
    subprocess.run([str(hostsim), str(n_fft), str(hop), "128", "0", str(tmp_path / "w.f32"), str(tmp_path / "o.f32")], check=True)
    got = np.fromfile(tmp_path / "o.f32", np.float32).reshape(-1, 128).T
    if key:
        ref = golden_extraction[f"{key}_{i}"][0]
    else:
        p = restate.power_spectrogram(wav, n_fft, hop, np.float64)
        ref = restate.amplitude_to_db_power((p.T @ restate.melscale_fbanks_htk(n_fft // 2 + 1, 128)).T)
    assert got.shape == ref.shape
    assert np.max(np.abs(got - ref)) < 1e-3          # dB, north_star tolerance


def test_kernel_phase_functions_on_host_gradient_stream(hostsim, golden_extraction, tmp_path):
    from oracle import restate
    wav = golden_extraction["wav3"]
    wav.tofile(tmp_path / "w.f32")
    subprocess.run([str(hostsim), "400", "200", "128", "1", str(tmp_path / "w.f32"), str(tmp_path / "o.f32")], check=True)
    got = np.fromfile(tmp_path / "o.f32", np.float32).reshape(-1, 128).T
    g = restate.waveform_gradient(wav, 1.0).astype(np.float64)
    p = restate.power_spectrogram(g, 400, 200, np.float64)
    ref = restate.amplitude_to_db_power((p.T @ restate.melscale_fbanks_htk(201, 128)).T)
    assert np.max(np.abs(got - ref)) < 1e-3


@pytest.fixture(scope="module")
def melprog(tmp_path_factory):
    exe = tmp_path_factory.mktemp("melprog") / "mel_program"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), str(REPO / "tests" / "hostsim" / "mel_program.cpp"), "-o", str(exe)],
                   check=True)
    return exe


@pytest.mark.parametrize("n_fft", [400, 800, 1600])
@pytest.mark.parametrize("n_mels", [1, 2, 5, 31, 32, 33, 40, 64, 100, 128, 200, 256, 512])
def test_mel_gather_program_encodes_the_filterbank(melprog, n_fft, n_mels):
    """The per-lane mel gather program (csrc/tables.h) holds every non-zero weight of melscale_fbanks exactly once, idle
    slots read a zero slot, and falling = 1/4 - rising for every entry (what the unrolled kernel path relies on)."""
    r = subprocess.run([str(melprog), str(n_fft), str(n_mels)], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0, f"mel_program exit code {r.returncode}"
    tag, steps, wavefronts, head = r.stdout.split()
    assert tag == "ok"
    if n_mels == 128:                                    # the reference's filterbank: the schedule stays near conflict free
        assert int(wavefronts) <= 1.25 * 2 * int(steps)


def test_fast_mel_step_counts_match_the_compiled_constants(melprog):
    """FastMel<R> in extract_core.cuh (compile-time step counts of the unrolled 128-band path) vs the built program."""
    import re
    src = (CSRC / "extract_core.cuh").read_text()
    for n_fft, R in ((400, 8), (800, 16), (1600, 32)):
        m = re.search(rf"FastMel<{R}> \{{ static constexpr int head = (\d+), s0 = (\d+), s1 = (\d+), s2 = (\d+), s3 = (\d+);", src)
        assert m, R
        head, *s = map(int, m.groups())
        out = subprocess.run([str(melprog), str(n_fft), "128"], stdout=subprocess.PIPE, text=True, check=True).stdout.split()
        assert int(out[1]) == sum(s) and int(out[3]) == head


def test_dropin_state_dict_keys_match_reference():
    import json
    from speech_emotion_privacy_trust_b200 import dropin
    dropin.install()
    import baseline_models
    import cloak_models
    spec = json.loads((REPO / "tests" / "golden" / "state_dict_keys.json").read_text())

    def keys(m):
        return {k: list(v.shape) for k, v in m.state_dict().items()}
    for cls in ("two_d_cnn_lstm", "deep_two_d_cnn_lstm"):
        for att in (None, "self_att"):
            m = getattr(baseline_models, cls)(1, 128, 5, lstm_hidden_size=64, num_layers_lstm=2, pred="emotion",
                                              bidirectional=True, rnn_cell="gru", global_feature=0, att=att)
            assert keys(m) == spec[f"{cls}|att={att}"]
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0)
    noise = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cpu")
    assert keys(cloak_models.two_d_cnn_lstm_syn(mk("emotion"), noise)) == spec["two_d_cnn_lstm_syn"]
    noise = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cpu")
    grl = cloak_models.two_d_cnn_lstm_syn_with_grl(mk("emotion"), mk("gender"), noise, 0.1)
    assert keys(grl) == spec["two_d_cnn_lstm_syn_with_grl"]
    assert float(noise.rhos.detach().mean()) == -2.0 and noise.locs.shape == (1, 200, 128)
    assert all(not p.requires_grad for p in grl.original_model.parameters())
    assert isinstance(grl.gender_model.conv[0], sys.modules["reversal_gradient"].GradientReversal)
    with pytest.raises(ValueError, match="Unsupported RNN Cell"):
        baseline_models.two_d_cnn_lstm(1, 128, 5, rnn_cell="rnn")
    # scales(): sigma = (1 + tanh(-2)) / 2 * (max - min) + min   (cloak_models.py:41-43)
    assert torch.allclose(noise.scales(), torch.full((1, 200, 128), (1 + np.tanh(-2.0)) / 2 * 9.99 + 0.01), atol=1e-6)


def test_cpu_classifier_forward_shapes():
    from speech_emotion_privacy_trust_b200 import dropin
    dropin.install()
    import baseline_models
    x = torch.randn(2, 1, 200, 128)
    m = baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred="multitask", global_feature=0).eval()
    e, g = m(x)
    assert e.shape == (2, 4) and g.shape == (2, 2)
    d = baseline_models.deep_two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred="gender", global_feature=0).eval()
    assert d(x).shape == (2, 2)
    a = baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred="emotion", global_feature=0, att="self_att").eval()
    assert a(x).shape == (2, 4)
