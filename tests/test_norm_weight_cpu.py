"""The training-window multiplicity of csrc/norm_weight.cuh -- the weight of every frame in the per-speaker statistics,
shared by utt_partial_kernel (frame_weight), utt_partial128_kernel and the backward (frame_weight_fast) -- built for the
host and compared with oracle.norm.frame_multiplicity for every frame of every utterance length up to 3000 frames."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import norm as onorm

REPO = Path(__file__).resolve().parents[1]

# (win_len, shift_len, longest utterance): the reference's 200/50; a shift that does not divide the window; a tiny
# window; a shift longer than the window (frames between windows have weight 0); shift == window; shift 1
WINDOWS = [(200, 50, 3000), (100, 30, 3000), (7, 3, 3000), (50, 80, 3000), (200, 200, 3000), (10, 1, 600)]


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = tmp_path_factory.mktemp("norm_weight") / "norm_weight"
    subprocess.run(["g++", "-O2", "-std=c++17", "-D__device__=", "-D__forceinline__=inline",
                    "-I", str(REPO / "speech_emotion_privacy_trust_b200" / "csrc"),
                    str(REPO / "tests" / "hostsim" / "norm_weight.cpp"), "-o", str(out)], check=True)
    return out


@pytest.mark.parametrize("win,shift,t_max,whole", [(*w, False) for w in WINDOWS] + [(200, 50, 3000, True)])
def test_frame_weight_matches_oracle(exe, tmp_path, win, shift, t_max, whole):
    path = tmp_path / "w.bin"
    subprocess.run([str(exe), "weights", str(win), str(shift), str(t_max), str(int(whole)), str(path)], check=True)
    raw = np.fromfile(path, np.int32)
    n = t_max * (t_max + 1) // 2
    assert raw.size == 2 * n
    slow, fast = raw[:n], raw[n:]
    want = np.concatenate([onorm.frame_multiplicity(T, whole, win, shift) for T in range(1, t_max + 1)])
    bad_slow, bad_fast = np.flatnonzero(slow != want), np.flatnonzero(fast != want)
    assert bad_slow.size == 0, f"frame_weight differs at {bad_slow.size} frames"
    assert bad_fast.size == 0, f"frame_weight_fast differs at {bad_fast.size} frames"


def test_div_floor_small_exact_below_2_pow_22(exe):
    divisors = list(range(1, 65)) + [80, 100, 127, 128, 160, 199, 200, 255, 256, 400, 1000, 1023, 1024, 3000, 4097,
                                     65535, (1 << 21) + 1, (1 << 22) - 1]
    r = subprocess.run([str(exe), "div", *map(str, divisors)], check=True, stdout=subprocess.PIPE, text=True)
    assert r.stdout.strip().endswith("mismatches 0"), r.stdout
