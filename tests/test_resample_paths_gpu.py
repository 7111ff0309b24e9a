"""The sinc resampler on every kernel path the C ABI reaches, against float64 (tests/test_resample_paths_cpu.py names the
paths and checks that each rate pair below still takes its own).

The reference.  Every output sample y[m * up + j] = sum_k w[j][k] * x[m * orig + k_lo[j] + k - width] is recomputed in
float64 from the library's own fp32 rows (tests/hostsim/resample_rows.cpp) and the fp32 input, zero padded outside the
utterance.  Both kernels evaluate that sum as one FMA chain over ascending taps; the tiled kernel's extra window taps
have zero weight and its pads are zeros, so they add exact zeros.  With T stored taps the chain is within
gamma_T * sum_k |w_k x_k| of the exact sum, gamma_T = T u / (1 - T u), u = 2^-24; that is the bound asserted here.

Tiled against simple.  With finite input the two kernels do the same FMAs in the same order, so their outputs must be
identical.  SEPT_RESAMPLE_SIMPLE=1 (read once per process) forces the simple kernel: a child process runs every case of
the tiled pairs with it and writes its outputs to one file.

The 64-bit case needs about 12 GB of device memory."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

from speech_emotion_privacy_trust_b200 import _lib
from test_resample_paths_cpu import (CLASSES, REJECTED, SIMPLE, build_resample_shape, class_of, length_rule,
                                     resample_shape)

pytestmark = pytest.mark.gpu

REPO = Path(__file__).resolve().parents[1]
CSRC = REPO / "speech_emotion_privacy_trust_b200" / "csrc"
SMS = 148                                   # the launcher sizes the tiled kernel's persistent grid for a B200's SMs
RUN = sorted(p for p, c in CLASSES.items() if c[1] != REJECTED)
TILED = [p for p in RUN if CLASSES[p][1] != SIMPLE]
CHUNK_WALK = [(44100, 16000), (16000, 44100)]      # two CTAs per SM (<43>) and three per SM (441 phases)
BIG = (16000, 44100, 779_366_400)            # output 2 148 128 768 samples: past 2^31, 128 past the exact ceil
WORST = {}                                   # class -> largest |y - r| / bound


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print(f"\nworst |y - r| / (gamma_T sum|w x|) per class on {torch.cuda.get_device_name()}:")
    for cls, w in sorted(WORST.items()):
        print(f"  {cls}: {w:.3g}")


# ---- cases (built the same way in this process and in the child that forces the simple kernel) ----------------------

def make_case(lengths, seed, lead=5, tail=9, align=0, device="cuda"):
    """Utterances of the given lengths back to back after `lead` and before `tail` samples of NaN, the whole buffer at
    storage offset `align` floats; returns (x, in_off) with in_off[0] = lead."""
    lengths = np.asarray(lengths, dtype=np.int64)
    in_off = np.concatenate([[0], np.cumsum(lengths)]) + lead
    g = torch.Generator(device=device).manual_seed(seed)
    total = int(in_off[-1]) + tail
    store = torch.full((total + 4,), float("nan"), device=device)
    x = store[align:align + total]
    x[lead:int(in_off[-1])] = 0.3 * torch.randn(int(in_off[-1]) - lead, generator=g, device=device)
    return x, in_off


def edge_lengths(shape, rng):
    """Ragged edge lengths of one rate pair; empty utterances first, last and consecutive."""
    orig, up, width, rows = shape["orig"], shape["up"], shape["width"], max(shape["rows_per_cta"], 4)
    pair = (shape["orig_freq"], shape["new_freq"])
    ls = {1, 2, width - 1, width, width + 1, orig - 1, orig, orig + 1, 2 * orig - 1, 2 * orig + 1, 5 * orig - 1,
          5 * orig + 1}
    # outputs that end inside a phase group: n_out % up not a multiple of 4, one of each residue
    cand = np.arange(3 * orig, 7 * orig, dtype=np.int64)
    r = length_rule(cand, *pair) % up % 4
    for res in (1, 2, 3):
        hit = cand[r == res]
        if hit.size:
            ls.add(int(hit[len(hit) // 2]))
    # long enough for chunks away from both ends: the interior cp.async fill
    n_long = 3 * rows * orig + 2 * width + 123
    ls |= {n_long, int(rng.integers(n_long, 2 * n_long))}
    ls = sorted(n for n in ls if n > 0)
    rng.shuffle(ls)
    h = len(ls) // 2
    return [0] + ls[:h] + [0, 0] + ls[h:] + [0]


def short_lengths(shape, rng):
    """20 000 utterances of 0-60 samples (0-4 where an input sample makes more than 8 outputs)."""
    hi = 60 if shape["up"] <= 8 * shape["orig"] else 4
    return rng.integers(0, hi + 1, 20_000).tolist()


def chunk_lengths(shape, rng):
    """A batch in which every worker of the persistent grid walks at least four chunks."""
    orig, up = shape["orig"], shape["up"]
    per_cta = shape["rows_per_cta"] * up
    want = 4 * 2 * SMS * shape["ctas_per_sm"] * per_cta * 1.1
    ls, out = [], 0
    while out < want:
        n = int(rng.integers(shape["orig_freq"] // 2, 3 * shape["orig_freq"]))
        ls.append(n)
        out += n * up // orig
    return ls


def permuted(x, in_off, perm, lead=5):
    """The same utterances in the order `perm`, in a fresh NaN-padded buffer."""
    parts = [x[in_off[u]:in_off[u + 1]] for u in perm]
    lengths = np.array([len(p) for p in parts], dtype=np.int64)
    off = np.concatenate([[0], np.cumsum(lengths)]) + lead
    y = torch.full((int(off[-1]) + 7,), float("nan"), device=x.device)
    for u, p in enumerate(parts):
        y[off[u]:off[u + 1]] = p
    return y, off


def run(x, in_off, pair, guard=64):
    """sept_resample_f32 into a NaN-filled output with a guard tail: every output sample must be written, and nothing
    past the end.  Returns (y, out_off)."""
    n = len(in_off) - 1
    out_off = np.zeros(n + 1, dtype=np.int64)
    _lib.call("sept_resample_layout", in_off.ctypes.data, n, pair[0], pair[1], out_off.ctypes.data)
    total = int(out_off[-1])
    out = torch.full((total + guard,), float("nan"), device=x.device)
    d_in, d_out = torch.from_numpy(in_off).to(x.device), torch.from_numpy(out_off).to(x.device)
    _lib.launch("sept_resample_f32", x, d_in, d_out, n, total, pair[0], pair[1], out, device=x.device)
    assert not torch.isnan(out[:total]).any().item(), (pair, "an output sample was not written or is NaN")
    assert torch.isnan(out[total:]).all().item(), (pair, "a write past the output")
    return out[:total], out_off


def big_windows(out_len):
    """Output windows of the 64-bit case: around sample 2^31 and the tail, which holds the samples past the exact
    ceil."""
    return [(2 ** 31 - 3000, 2 ** 31 + 3000), (out_len - 4000, out_len)]


def big_case(device="cuda"):
    orig_freq, new_freq, n = BIG
    g = torch.Generator(device=device).manual_seed(31)
    x = 0.3 * torch.randn(n, generator=g, device=device)
    return x, np.array([0, n], dtype=np.int64)


def all_cases(shapes, pairs):
    """{name: (pair, x, in_off)} of every tiled-vs-simple comparison; deterministic."""
    cases = {}
    for pair in pairs:
        s = shapes[pair]
        rng = np.random.default_rng(pair[0] * 7 + pair[1])
        cases[f"{pair}/edge"] = (pair, *make_case(edge_lengths(s, rng), seed=pair[0] + pair[1]))
        cases[f"{pair}/short"] = (pair, *make_case(short_lengths(s, rng), seed=pair[0] + 2 * pair[1]))
        if pair in CHUNK_WALK:
            cases[f"{pair}/chunks"] = (pair, *make_case(chunk_lengths(s, rng), seed=pair[0] + 3 * pair[1]))
    return cases


def simple_child(shapes_json, out_path):
    """Run in a child process with SEPT_RESAMPLE_SIMPLE=1: the simple kernel's output of every case, and of the 64-bit
    case's windows, into one file."""
    raw = json.loads(Path(shapes_json).read_text())
    shapes = {tuple(v["pair"]): v["shape"] for v in raw}
    res = {}
    for name, (pair, x, in_off) in all_cases(shapes, [p for p in shapes if p in TILED]).items():
        res[name] = run(x, in_off, pair)[0].cpu()
        del x
    x, in_off = big_case()
    y, out_off = run(x, in_off, BIG[:2])
    for lo, hi in big_windows(int(out_off[-1])):
        res[f"big/{lo}"] = y[lo:hi].cpu()
    torch.save(res, out_path)


# ---- float64 reference ------------------------------------------------------------------------------------------------

def load_rows(exe_rows, tmp, pair, shape):
    raw_path = tmp / f"rows_{shape['orig']}_{shape['up']}.bin"
    subprocess.run([str(exe_rows), str(shape["orig"]), str(shape["up"]), str(raw_path)], check=True)
    raw = np.fromfile(raw_path, np.int32)
    width, taps = int(raw[0]), int(raw[1])
    up = shape["up"]
    assert (width, taps) == (shape["width"], shape["taps"])
    return {"orig": shape["orig"], "up": up, "width": width, "taps": taps, "k_lo": raw[2:2 + up].astype(np.int64),
            "rows": raw[2 + up:].view(np.float32).reshape(up, taps).astype(np.float64)}


def ref64(tab, x_host, x_base, in_off, out_off, g):
    """(float64 sum, sum of |products|) of output samples g; x_host[i - x_base] is input sample i of the buffer."""
    orig, up, width, taps, k_lo, rows = (tab[k] for k in ("orig", "up", "width", "taps", "k_lo", "rows"))
    g = np.asarray(g, dtype=np.int64)
    u = np.searchsorted(out_off, g, side="right") - 1
    o = g - out_off[u]
    m, j = o // up, o % up
    i0 = m * orig + k_lo[j] - width
    n_in = in_off[u + 1] - in_off[u]
    r, a = np.empty(len(g)), np.empty(len(g))
    step = max(1, 2_000_000 // taps)
    for s in range(0, len(g), step):
        sl = slice(s, s + step)
        idx = i0[sl, None] + np.arange(taps)
        valid = (idx >= 0) & (idx < n_in[sl, None])
        src = np.where(valid, in_off[u[sl], None] + idx - x_base, 0)
        xv = np.where(valid, x_host[src].astype(np.float64), 0.0)
        p = rows[j[sl]] * xv
        r[sl], a[sl] = p.sum(axis=1), np.abs(p).sum(axis=1)
    return r, a


def check_bound(cls, tab, y, r, a):
    T = tab["taps"]
    gamma = T * 2.0 ** -24 / (1 - T * 2.0 ** -24)
    err = np.abs(np.asarray(y, dtype=np.float64) - r)
    bound = gamma * a
    bad = np.flatnonzero(err > bound)
    assert bad.size == 0, (cls, [(int(i), float(err[i]), float(bound[i])) for i in bad[:5]])
    pos = bound > 0
    if pos.any():
        WORST[cls] = max(WORST.get(cls, 0.0), float(np.max(err[pos] / bound[pos])))


def check_all(cls, tab, x, in_off, y, out_off, g=None):
    """Float64 bound on output samples g (all of them by default)."""
    g = np.arange(int(out_off[-1])) if g is None else g
    r, a = ref64(tab, x.cpu().numpy(), 0, in_off, out_off, g)
    check_bound(cls, tab, y.cpu().numpy()[g], r, a)


# ---- fixtures -----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def tools(tmp_path_factory):
    d = tmp_path_factory.mktemp("resample_tools")
    shape_exe = build_resample_shape(d)
    rows_exe = d / "resample_rows"
    subprocess.run(["g++", "-O1", "-std=c++17", "-I", str(CSRC), str(REPO / "tests" / "hostsim" / "resample_rows.cpp"),
                    "-o", str(rows_exe)], check=True)
    shapes, tabs = {}, {}
    for pair in RUN:
        class_of(shape_exe, *pair)
        s = resample_shape(shape_exe, *pair)
        s.update(orig_freq=pair[0], new_freq=pair[1])
        shapes[pair] = s
        tabs[pair] = load_rows(rows_exe, d, pair, s)
    shapes_json = d / "shapes.json"
    shapes_json.write_text(json.dumps([{"pair": list(p), "shape": s} for p, s in shapes.items()]))
    return d, shapes, tabs, shapes_json


@pytest.fixture(scope="module")
def simple_out(tools):
    """The simple kernel's outputs of every tiled-pair case, from a child process with SEPT_RESAMPLE_SIMPLE=1."""
    d, _, _, shapes_json = tools
    out = d / "simple.pt"
    code = (f"import sys; sys.path[:0] = [{str(REPO / 'tests')!r}, {str(REPO)!r}]\n"
            "import test_resample_paths_gpu as t\n"
            f"t.simple_child({str(shapes_json)!r}, {str(out)!r})\n")
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, SEPT_RESAMPLE_SIMPLE="1"),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    return torch.load(out)


@pytest.fixture(scope="module")
def cases(tools):
    _, shapes, _, _ = tools
    return all_cases(shapes, TILED)


def cls_name(pair):
    return f"{CLASSES[pair][0]} {pair[0]}->{pair[1]}"


# ---- tests ------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pair", RUN, ids=lambda p: f"{p[0]}-{p[1]}")
def test_edge_lengths_outside_nan_alignment_and_batch_invariance(tools, pair):
    """Ragged edge lengths with NaN outside every utterance (before the first, after the last): float64 bound on every
    output sample; the same buffer at storage offsets 0-3 floats, each utterance alone and the batch shuffled: bit
    identical."""
    _, shapes, tabs, _ = tools
    s, tab = shapes[pair], tabs[pair]
    lengths = edge_lengths(s, np.random.default_rng(pair[0] * 7 + pair[1]))
    x, in_off = make_case(lengths, seed=pair[0] + pair[1])
    y, out_off = run(x, in_off, pair)
    assert np.array_equal(np.diff(out_off), length_rule(lengths, *pair))
    check_all(cls_name(pair), tab, x, in_off, y, out_off)
    for align in (1, 2, 3):
        xa, _ = make_case(lengths, seed=pair[0] + pair[1], align=align)
        assert xa.data_ptr() % 16 == 4 * align
        assert torch.equal(run(xa, in_off, pair)[0], y), align
    for u in range(len(lengths)):
        xu = x[in_off[u]:in_off[u + 1]].clone()
        yu, _ = run(xu, np.array([0, lengths[u]], dtype=np.int64), pair)
        assert torch.equal(yu, y[out_off[u]:out_off[u + 1]]), u
    perm = np.random.default_rng(1).permutation(len(lengths))
    xp, offp = permuted(x, in_off, perm)
    yp, outp = run(xp, offp, pair)
    for k, u in enumerate(perm):
        assert torch.equal(yp[outp[k]:outp[k + 1]], y[out_off[u]:out_off[u + 1]]), u


@pytest.mark.parametrize("pair", RUN, ids=lambda p: f"{p[0]}-{p[1]}")
def test_many_short_utterances(tools, pair):
    """20 000 utterances of a few samples each, many to a chunk: float64 bound on a seeded subset, shuffled batch bit
    identical."""
    _, shapes, tabs, _ = tools
    s, tab = shapes[pair], tabs[pair]
    rng = np.random.default_rng(pair[0] * 7 + pair[1])
    edge_lengths(s, rng)                                     # the same draws as all_cases()
    lengths = short_lengths(s, rng)
    x, in_off = make_case(lengths, seed=pair[0] + 2 * pair[1])
    y, out_off = run(x, in_off, pair)
    assert np.array_equal(np.diff(out_off), length_rule(lengths, *pair))
    pick = np.random.default_rng(2).choice(len(lengths), 300, replace=False)
    g = np.concatenate([np.arange(out_off[u], out_off[u + 1]) for u in pick])
    check_all(cls_name(pair), tab, x, in_off, y, out_off, g)
    perm = np.random.default_rng(3).permutation(len(lengths))
    xp, offp = permuted(x, in_off, perm)
    yp, outp = run(xp, offp, pair)
    y_host, yp_host = y.cpu().numpy(), yp.cpu().numpy()
    for k, u in enumerate(perm):
        assert np.array_equal(yp_host[outp[k]:outp[k + 1]], y_host[out_off[u]:out_off[u + 1]]), u


@pytest.mark.parametrize("pair", CHUNK_WALK, ids=lambda p: f"{p[0]}-{p[1]}")
def test_multi_chunk_walk(tools, pair):
    """Every worker of the persistent grid walks at least four chunks: shuffled batch bit identical on all of it, float64
    bound on a seeded subset of utterances."""
    _, shapes, tabs, _ = tools
    s, tab = shapes[pair], tabs[pair]
    rng = np.random.default_rng(pair[0] * 7 + pair[1])
    edge_lengths(s, rng), short_lengths(s, rng)
    lengths = chunk_lengths(s, rng)
    x, in_off = make_case(lengths, seed=pair[0] + 3 * pair[1])
    y, out_off = run(x, in_off, pair)
    per_cta = s["rows_per_cta"] * s["up"]
    workers = 2 * SMS * s["ctas_per_sm"]
    assert -(-int(out_off[-1]) // per_cta) >= 4 * workers
    pick = np.random.default_rng(4).choice(len(lengths), 12, replace=False)
    g = np.concatenate([np.arange(out_off[u], out_off[u + 1]) for u in pick])
    check_all(f"{cls_name(pair)} chunk walk", tab, x, in_off, y, out_off, g)
    perm = np.random.default_rng(5).permutation(len(lengths))
    xp, offp = permuted(x, in_off, perm)
    yp, outp = run(xp, offp, pair)
    for k, u in enumerate(perm):
        assert torch.equal(yp[outp[k]:outp[k + 1]], y[out_off[u]:out_off[u + 1]]), u


def test_tiled_equals_simple(tools, cases, simple_out):
    """Every case of every tiled pair, bit for bit against the simple kernel."""
    for name, (pair, x, in_off) in cases.items():
        y, _ = run(x, in_off, pair)
        assert torch.equal(y.cpu(), simple_out[name]), name


def test_output_past_2_31_samples(tools, simple_out):
    """One 16 -> 44.1 kHz utterance of 779 366 400 samples: 2 148 128 768 output samples, 128 of them past the exact
    ceil.  The length is torchaudio's; windows around sample 2^31 and the tail are within the float64 bound and equal
    the simple kernel's."""
    _, _, tabs, _ = tools
    orig_freq, new_freq, n = BIG
    tab = tabs[(orig_freq, new_freq)]
    x, in_off = big_case()
    y, out_off = run(x, in_off, (orig_freq, new_freq))
    out_len = int(out_off[-1])
    assert out_len == int(length_rule([n], orig_freq, new_freq)[0]) == 2_148_128_768
    assert out_len - (-(-441 * n // 160)) == 128
    for lo, hi in big_windows(out_len):
        g = np.arange(lo, hi)
        m = g // tab["up"]
        i_lo = max(0, int(m.min() * tab["orig"] - tab["width"]))
        i_hi = min(n, int(m.max() * tab["orig"] + tab["k_lo"].max() - tab["width"] + tab["taps"]))
        r, a = ref64(tab, x[i_lo:i_hi].cpu().numpy(), i_lo, in_off, out_off, g)
        yw = y[lo:hi].cpu()
        check_bound("64-bit indices 16000->44100", tab, yw.numpy(), r, a)
        assert torch.equal(yw, simple_out[f"big/{lo}"]), lo
