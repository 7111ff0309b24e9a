"""The sinc resampler's host side without a device: the output length rule against torchaudio itself, the kernel each
rate pair takes (computed by the library's own host functions, tests/hostsim/resample_shape.cpp), and the argument
checks of sept_resample_layout, sept_resample_f32 and sept_pcm16_to_f32.

Output length.  torchaudio's _apply_sinc_resample_kernel, which the reference's Resample calls, cuts each utterance at
ceil(torch.as_tensor(new * length / orig)) with gcd-reduced rates: the Python float quotient is rounded to float32 (the
default dtype) before the ceil, so for about 1 % of lengths at 44.1 -> 16 kHz it is one less than the exact ceil, and
for long utterances it can be one more.  The library and oracle/restate.py must cut where torchaudio does.

Kernel paths.  A rate pair takes the tiled kernel when its weight table and two stages fit 112 KB of shared memory
(three CTAs per SM at 72 KB or less; the unrolled <43> instantiation at the 44.1 -> 16 kHz tap count), the simple
one-thread-per-sample kernel above that, and is refused beyond 4096 phases.  The named pairs below are the ones
tests/test_resample_paths_gpu.py runs, each checked here to still take the path it is meant to reach."""
import ctypes
import math
import subprocess
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import restate
from speech_emotion_privacy_trust_b200 import _lib
from test_extraction_paths_cpu import cuda_include

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"

FIELDS = ("orig_freq", "orig", "up", "width", "taps", "n_groups", "tg", "group_span", "base_span", "rows_per_cta", "stage_floats",
          "smem", "kernel", "ctas_per_sm")
REJECTED, SIMPLE, TILED, TILED43 = -1, 0, 1, 2
TILED_MAX_SMEM, TILED_3CTA_SMEM = 112 * 1024, 72 * 1024
SEPT_OK = 0

# (orig_freq, new_freq) -> (class, kernel, CTAs per SM, rows per CTA, tg)
CLASSES = {
    (44100, 16000): ("tiled43", TILED43, 2, 16, 43),
    (48000, 16000): ("one_group", TILED, 3, 1024, 37),
    (8000, 16000): ("one_group", TILED, 3, 1024, 15),
    (16000, 48000): ("one_group", TILED, 3, 1024, 15),
    (12000, 16000): ("one_group", TILED, 3, 1024, 17),
    (16000, 44100): ("up_not_mult4", TILED, 3, 8, 15),
    (192000, 16000): ("mg_fit", TILED, 2, 744, 145),
    (11025, 16000): ("rows4_3cta", TILED, 3, 4, 17),
    (22050, 16000): ("tiled_2cta", TILED, 2, 12, 23),
    (16000, 11025): ("tiled_2cta", TILED, 2, 8, 23),
    (176400, 16000): ("tiled_2cta", TILED, 2, 16, 169),
    (999, 1000): ("simple", SIMPLE, 0, 4, 17),
    (1000, 999): ("simple", SIMPLE, 0, 4, 17),
    (1, 4096): ("simple", SIMPLE, 0, 4, 15),
    (4095, 4096): ("simple", SIMPLE, 0, 4, 17),
    (4096, 1): ("simple", SIMPLE, 0, 4, 49649),
    (15999, 16000): ("rejected", REJECTED, 0, 0, 0),
    (4097, 4096): ("rejected", REJECTED, 0, 0, 0),
}

USUAL_RATES = (8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000, 88200, 96000, 176400, 192000)


def build_resample_shape(out_dir: Path) -> Path:
    exe = out_dir / "resample_shape"
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", str(CSRC), "-I", str(cuda_include()),
                    str(REPO / "tests" / "hostsim" / "resample_shape.cpp"), "-o", str(exe)], check=True)
    return exe


def resample_shape(exe: Path, orig_freq: int, new_freq: int) -> dict:
    """The launch configuration of one rate pair (FIELDS without orig_freq)."""
    out = subprocess.run([str(exe), str(orig_freq), str(new_freq)], check=True, capture_output=True, text=True).stdout
    words = out.split()
    return {k: int(v) for k, v in zip(words[::2], words[1::2])}


def classes_of(s: dict) -> set:
    """Every class of the table above that a launch configuration belongs to."""
    if s["kernel"] == REJECTED:
        return {"rejected"}
    if s["kernel"] == SIMPLE:
        return {"simple"}
    c = {"tiled43"} if s["kernel"] == TILED43 else set()
    if s["n_groups"] == 1 and s["rows_per_cta"] == 1024:
        c.add("one_group")
    if s["up"] % 4 and s["n_groups"] > 1:
        c.add("up_not_mult4")
    if s["rows_per_cta"] < 4 * max(1, 256 // s["n_groups"]):
        c.add("mg_fit")
    if s["rows_per_cta"] == 4 and s["ctas_per_sm"] == 3:
        c.add("rows4_3cta")
    if s["ctas_per_sm"] == 2:
        c.add("tiled_2cta")
    return c


def class_of(exe: Path, orig_freq: int, new_freq: int) -> str:
    """The class a GPU test names for a rate pair, asserted through the helper."""
    s = resample_shape(exe, orig_freq, new_freq)
    name = CLASSES[(orig_freq, new_freq)][0]
    assert name in classes_of(s), (orig_freq, new_freq, s)
    return name


# ---- output length ------------------------------------------------------------------------------------------------

def length_rule(n: np.ndarray, orig_freq: int, new_freq: int) -> np.ndarray:
    """torchaudio's cut, vectorised: ceil(float32(up * n / orig)) with the quotient in float64 (exact products below
    2^53, so Python's int / int), at most the (n // orig + 1) * up samples of its conv1d."""
    g = math.gcd(orig_freq, new_freq)
    orig, up = orig_freq // g, new_freq // g
    n = np.asarray(n, dtype=np.int64)
    assert np.all(up * n < 2 ** 53)
    cut = np.ceil(((up * n).astype(np.float64) / orig).astype(np.float32)).astype(np.int64)
    return np.minimum(cut, (n // orig + 1) * up)


def layout(lengths, orig_freq: int, new_freq: int) -> np.ndarray:
    in_off = np.concatenate([[0], np.cumsum(np.asarray(lengths, dtype=np.int64))]).astype(np.int64)
    out_off = np.zeros_like(in_off)
    _lib.call("sept_resample_layout", in_off.ctypes.data, len(in_off) - 1, orig_freq, new_freq, out_off.ctypes.data)
    return np.diff(out_off)


RULE_PAIRS = ((44100, 16000), (22050, 16000), (16000, 44100), (44100, 48000), (48000, 16000))


@pytest.mark.parametrize("orig_freq,new_freq", RULE_PAIRS)
def test_layout_is_the_length_rule_for_every_length(orig_freq, new_freq):
    n = np.arange(0, 3_000_001, dtype=np.int64)
    want = length_rule(n, orig_freq, new_freq)
    got = layout(n, orig_freq, new_freq)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, [(int(n[i]), int(got[i]), int(want[i])) for i in bad[:5]]
    exact = -(-(new_freq // math.gcd(orig_freq, new_freq)) * n // (orig_freq // math.gcd(orig_freq, new_freq)))
    assert np.all(np.abs(want - exact) <= 1)


@pytest.mark.parametrize("n,orig_freq,new_freq,want", [(180697, 44100, 16000, 65559), (47561, 16000, 44100, 131090),
                                                       (120427, 44100, 48000, 131077),
                                                       (6087520, 16000, 44100, 16778728)])
def test_layout_cuts_where_torchaudio_does(n, orig_freq, new_freq, want):
    """The lengths where the exact ceil and torchaudio differ, the last one longer than the exact ceil."""
    assert layout([n], orig_freq, new_freq)[0] == want == length_rule([n], orig_freq, new_freq)[0]
    assert restate.resample_length(n, orig_freq, new_freq) == want


def torchaudio_cases(orig_freq: int, new_freq: int, rng) -> list:
    """The first ten lengths where the float32 rule and the exact ceil differ, and random lengths."""
    n = np.arange(0, 400_000, dtype=np.int64)
    g = math.gcd(orig_freq, new_freq)
    exact = -(-(new_freq // g) * n // (orig_freq // g))
    differ = n[length_rule(n, orig_freq, new_freq) != exact][:10]
    return sorted(set(differ.tolist()) | set(rng.integers(0, 200_000, 6).tolist()) | {0, 1, 2})


@pytest.mark.parametrize("orig_freq,new_freq", [p for p in RULE_PAIRS if p != (48000, 16000)])
def test_torchaudio_lengths(orig_freq, new_freq):
    from oracle import ref_port
    lengths = torchaudio_cases(orig_freq, new_freq, np.random.default_rng(orig_freq + new_freq))
    assert any(length_rule([n], orig_freq, new_freq)[0] != -(-new_freq * n // orig_freq) for n in lengths)
    lay = layout(lengths, orig_freq, new_freq)
    for n, want in zip(lengths, lay):
        got = ref_port.resample(torch.zeros(1, n), orig_freq, new_freq).shape[-1] if n else 0
        assert got == want, (n, got, want)
        assert restate.resample(np.zeros(n, np.float32), orig_freq, new_freq).shape == (want,)


def test_torchaudio_length_past_the_exact_ceil():
    """6 087 520 samples at 16 -> 44.1 kHz: torchaudio keeps one sample past the exact ceil; the layout, the oracle and
    torchaudio agree on it."""
    from oracle import ref_port
    n = 6_087_520
    x = np.random.default_rng(5).standard_normal(n).astype(np.float32) * 0.1
    ta = ref_port.resample(torch.from_numpy(x)[None], 16000, 44100)[0].numpy()
    assert ta.shape == (16_778_728,) == tuple(layout([n], 16000, 44100))
    ours = restate.resample(x, 16000, 44100)
    assert ours.shape == ta.shape
    assert np.max(np.abs(ours[-4:] - ta[-4:])) < 1e-6


# ---- kernel paths -------------------------------------------------------------------------------------------------

def sweep_pairs() -> np.ndarray:
    """All pairs of rates 1..64, every ordered pair of the usual rates and a seeded sample up to 4096 phases (and a few
    beyond)."""
    pairs = {(o, u) for o in range(1, 65) for u in range(1, 65)}
    pairs |= {(a, b) for a in USUAL_RATES for b in USUAL_RATES if a != b}
    rng = np.random.default_rng(4096)
    pairs |= {(int(o), int(u)) for o, u in rng.integers(1, 4097, (120, 2))}
    pairs |= {(int(o), int(u)) for o, u in rng.integers(1, 6000, (20, 2))}
    pairs |= set(CLASSES)
    return np.array(sorted(pairs), dtype=np.int32)


@pytest.fixture(scope="module")
def sweep(tmp_path_factory):
    d = tmp_path_factory.mktemp("resample_shape")
    exe = build_resample_shape(d)
    pairs = sweep_pairs()
    pairs.tofile(d / "pairs.i32")
    subprocess.run([str(exe), "list", str(d / "pairs.i32"), str(d / "shapes.i32")], check=True)
    rows = np.fromfile(d / "shapes.i32", dtype=np.int32).reshape(-1, len(FIELDS))
    assert len(rows) == len(pairs) and np.array_equal(rows[:, 0], pairs[:, 0])
    s = {k: rows[:, i].astype(np.int64) for i, k in enumerate(FIELDS)}
    s["new_freq"] = pairs[:, 1].astype(np.int64)
    return exe, s


def test_every_accepted_pair_resolves_to_a_kernel(sweep):
    _, s = sweep
    g = np.gcd(s["orig_freq"], s["new_freq"])
    assert np.array_equal(s["orig"], s["orig_freq"] // g) and np.array_equal(s["up"], s["new_freq"] // g)
    beyond = (s["orig"] > 4096) | (s["up"] > 4096)
    assert np.array_equal(s["kernel"] == REJECTED, beyond)
    assert beyond.any() and (~beyond).sum() > 2500
    assert set(np.unique(s["kernel"][~beyond])) == {SIMPLE, TILED, TILED43}


def test_tiled_kernel_only_within_its_shared_memory(sweep):
    _, s = sweep
    ok = s["kernel"] != REJECTED
    tiled = ok & (s["kernel"] != SIMPLE)
    assert np.array_equal(tiled, ok & (s["smem"] <= TILED_MAX_SMEM))
    assert np.array_equal(s["ctas_per_sm"][tiled] == 3, s["smem"][tiled] <= TILED_3CTA_SMEM)
    assert set(np.unique(s["ctas_per_sm"][tiled])) == {2, 3} and np.all(s["ctas_per_sm"][ok & ~tiled] == 0)
    assert np.array_equal(s["kernel"][tiled] == TILED43, s["tg"][tiled] == 43)
    # the shared memory the launcher asks for: weight table, group bases, two stages
    want = s["n_groups"] * s["tg"] * 16 + ((s["n_groups"] + 3) & ~3) * 4 + 2 * s["stage_floats"] * 4
    assert np.array_equal(s["smem"][ok], want[ok])


def test_tables_and_stage_hold_what_a_chunk_touches(sweep):
    _, s = sweep
    ok = s["kernel"] != REJECTED
    o = {k: v[ok] for k, v in s.items()}
    assert np.array_equal(o["n_groups"], (o["up"] + 3) // 4)
    assert np.all(o["tg"] % 2 == 1) and np.all(o["tg"] >= o["taps"] + o["group_span"])
    assert np.all(o["taps"] <= 2 * o["width"] + 4) and np.all(o["taps"] >= 1)
    assert np.all(o["rows_per_cta"] % 4 == 0) and np.all(o["rows_per_cta"] >= 4)
    # a chunk of rows_per_cta * up samples need not start on a row boundary: it touches rows_per_cta / 4 + 1 row quads;
    # the span is staged from the 16-byte boundary below it (up to 3 floats earlier) in whole float4s
    quads = o["rows_per_cta"] // 4 + 1
    widest = (4 * quads - 1) * o["orig"] + o["base_span"] + o["tg"] + 3
    assert np.all(o["stage_floats"] % 4 == 0) and np.all(o["stage_floats"] >= (widest + 3) // 4 * 4)


def test_every_class_is_reached(sweep):
    _, s = sweep
    seen = set()
    for i in range(len(s["orig"])):
        seen |= classes_of({k: int(v[i]) for k, v in s.items()})
    assert {c for c, *_ in CLASSES.values()} <= seen


@pytest.mark.parametrize("pair", sorted(CLASSES), ids=lambda p: f"{p[0]}-{p[1]}")
def test_named_pairs_keep_their_class(sweep, pair):
    exe, s = sweep
    name, kernel, ctas, rows, tg = CLASSES[pair]
    assert class_of(exe, *pair) == name
    got = resample_shape(exe, *pair)
    assert (got["kernel"], got["ctas_per_sm"]) == (kernel, ctas)
    if kernel != REJECTED:
        assert (got["rows_per_cta"], got["tg"]) == (rows, tg)
        if kernel != SIMPLE:
            assert got["smem"] <= TILED_MAX_SMEM
        else:
            assert got["smem"] > TILED_MAX_SMEM
    i = np.flatnonzero((s["orig_freq"] == pair[0]) & (s["new_freq"] == pair[1]))
    assert len(i) == 1 and all(int(s[k][i[0]]) == v for k, v in got.items())


# ---- C ABI checks without a device ---------------------------------------------------------------------------------

def _layout_rc(in_off, n_utts, orig_freq, new_freq, out=True):
    in_off = None if in_off is None else np.asarray(in_off, dtype=np.int64)
    out_off = np.zeros(max(n_utts, 0) + 1, dtype=np.int64)
    return _lib.lib().sept_resample_layout(None if in_off is None else in_off.ctypes.data, n_utts, orig_freq, new_freq,
                                           out_off.ctypes.data if out else None)


@pytest.mark.parametrize("args", [(None, 1, 44100, 16000), ([0, 5], -1, 44100, 16000), ([0, 5], 1, 0, 16000),
                                  ([0, 5], 1, 44100, 0), ([0, 5], 1, -44100, 16000), ([0, 5, 3], 2, 44100, 16000),
                                  ([0, (2 ** 53 - 1) // 160 + 1], 1, 44100, 16000)])
def test_layout_rejects_bad_arguments(args):
    assert _layout_rc(*args) == _lib.SEPT_E_BADARG
    assert "sept_resample_layout" in _lib.lib().sept_last_error().decode()


def test_layout_rejects_null_output_and_too_many_phases():
    assert _layout_rc([0, 5], 1, 44100, 16000, out=False) == _lib.SEPT_E_BADARG
    for pair in ((15999, 16000), (4097, 4096), (1, 4097)):
        assert _layout_rc([0, 5], 1, *pair) == _lib.SEPT_E_UNSUPPORTED, pair
        assert "4096" in _lib.lib().sept_last_error().decode()
    assert _layout_rc([0, (2 ** 53 - 1) // 160], 1, 44100, 16000) == SEPT_OK   # up * n just below 2^53
    assert _layout_rc([0, 5], 1, 4096, 4095) == SEPT_OK
    assert _layout_rc([0], 0, 44100, 16000) == SEPT_OK


def _bufs():
    b = {"x": (ctypes.c_float * 64)(), "in_off": (ctypes.c_int64 * 2)(0, 44), "out_off": (ctypes.c_int64 * 2)(0, 16),
         "y": (ctypes.c_float * 64)(), "pcm": (ctypes.c_int16 * 64)()}
    return b, {k: ctypes.addressof(v) for k, v in b.items()}


def _resample_rc(a, **kw):
    v = dict(a, n_utts=1, total_out=16, orig=44100, new=16000)
    v.update(kw)
    return _lib.lib().sept_resample_f32(v["x"], v["in_off"], v["out_off"], v["n_utts"], v["total_out"], v["orig"],
                                        v["new"], v["y"], None)


@pytest.mark.parametrize("bad", [dict(x=None), dict(in_off=None), dict(out_off=None), dict(y=None), dict(n_utts=-1),
                                 dict(total_out=-1), dict(orig=0), dict(new=0), dict(orig=-44100), dict(new=-16000)])
def test_resample_rejects_bad_arguments(bad):
    keep, a = _bufs()
    assert _resample_rc(a, **bad) == _lib.SEPT_E_BADARG
    assert "sept_resample_f32" in _lib.lib().sept_last_error().decode()


@pytest.mark.parametrize("pair", [(15999, 16000), (4097, 4096), (16000, 4097)])
def test_resample_rejects_too_many_phases(pair):
    keep, a = _bufs()
    assert _resample_rc(a, orig=pair[0], new=pair[1]) == _lib.SEPT_E_UNSUPPORTED
    assert "4096-phase" in _lib.lib().sept_last_error().decode()


def test_resample_empty_work_returns_before_any_launch():
    """n_utts == 0 or total_out == 0 is no work: OK without touching a device (on a machine without one, anything that
    reached the CUDA runtime would fail with SEPT_E_CUDA)."""
    keep, a = _bufs()
    assert _resample_rc(a, n_utts=0) == SEPT_OK
    assert _resample_rc(a, total_out=0) == SEPT_OK
    assert _resample_rc(a, n_utts=0, total_out=0, x=None, y=None) == SEPT_OK


def test_pcm16_argument_checks():
    keep, a = _bufs()
    lib = _lib.lib()
    assert lib.sept_pcm16_to_f32(None, 4, a["y"], None) == _lib.SEPT_E_BADARG
    assert lib.sept_pcm16_to_f32(a["pcm"], 4, None, None) == _lib.SEPT_E_BADARG
    assert lib.sept_pcm16_to_f32(a["pcm"], -1, a["y"], None) == _lib.SEPT_E_BADARG
    assert "sept_pcm16_to_f32" in lib.sept_last_error().decode()
    assert lib.sept_pcm16_to_f32(a["pcm"], 0, a["y"], None) == SEPT_OK
    assert lib.sept_pcm16_to_f32(None, 0, None, None) == SEPT_OK


def test_resample_fails_loudly_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("a device is present")
    keep, a = _bufs()
    assert _resample_rc(a) == _lib.SEPT_E_CUDA
    assert _lib.lib().sept_pcm16_to_f32(a["pcm"], 4, a["y"], None) == _lib.SEPT_E_CUDA
