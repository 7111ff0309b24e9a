"""Evaluation of a waveform cloak with fresh noise per utterance (sept_wave_cloak_eval_f32, WaveCloak.noisy_per_utterance,
evaluation.wave_cloak_evaluate) on the GPU.

The noisy audio is held bit for bit to the composition a user would write without the fused kernel: per-utterance noise
rows drawn by sept_cloak_fwd_f32(per_sample = 1) (through cloak_ops.cloak_forward_raw) at the same seed and counter,
then x + row[d_u][phase] in numpy float32.  The evaluator is held to the reference's window loop restated per utterance,
and two gloo ranks on one device to one GPU."""
import os
from datetime import timedelta

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import wave_cloak_order as order

pytestmark = pytest.mark.gpu

# shorter than, equal to and several periods; lengths that are not multiples of 4; empty utterances
LENGTHS = [3, 4, 5, 1, 43, 44, 45, 0, 88, 131, 999, 1000, 1001, 2003, 31999, 32000, 32001, 64005, 96003, 7]
LEAD, TRAIL = 5, 3                   # samples before the first (so utterances start at odd offsets) and after the last
PERIODS = [4, 44, 1000, 32000]       # 44 and 1000 are not multiples of 16
MN, MX = 1e-3, 0.05


def _batch(lengths=LENGTHS, lead=LEAD, trail=TRAIL, seed=0):
    from speech_emotion_privacy_trust_b200 import extraction
    off = np.concatenate([[lead], lead + np.cumsum(lengths)]).astype(np.int64)
    x = np.random.default_rng(seed).standard_normal(int(off[-1]) + trail).astype(np.float32)
    return extraction.RaggedAudio(torch.from_numpy(x).cuda(), off), x, off


def _layer(period, seed=0, mn=MN, mx=MX):
    from speech_emotion_privacy_trust_b200 import wave_cloak
    g = torch.Generator().manual_seed(seed)
    layer = wave_cloak.WaveCloak(mn, mx, period=period, locs=0.01 * torch.randn(period, generator=g)).cuda()
    with torch.no_grad():
        layer.rhos.add_(torch.randn(period, generator=g).cuda())
    return layer


def _rows(layer, n_rows, draw0):
    """Rows draw0 .. draw0 + n_rows - 1 of sept_cloak_fwd_f32(per_sample = 1, wf = L) at the layer's seed, as
    0 + (mu + sigma * eps): the noise a user would draw per utterance without the fused kernel."""
    from speech_emotion_privacy_trust_b200 import cloak_ops, wave_cloak
    L = layer.period
    counter = torch.tensor([draw0], dtype=torch.int64, device="cuda")
    out, _, _ = cloak_ops.cloak_forward_raw(torch.zeros(n_rows * L, device="cuda"), layer.locs.detach(),
                                            layer.rhos.detach(), None, None, torch.initial_seed(), 0, wave_cloak.EPS_STD,
                                            layer.min_scale, layer.max_scale, draw=counter, per_sample=True)
    return out.view(n_rows, L).cpu().numpy()


def _expected(x, off, rows, row_of_utt):
    """x + rows[row_of_utt[u]][phase] over every utterance sample, in float32; samples outside every utterance are x."""
    ph = order.phase_of(off, len(x), rows.shape[1])
    s = np.nonzero(ph >= 0)[0]
    u = np.searchsorted(off, s, side="right") - 1
    y = x.copy()
    y[s] = x[s] + rows[np.asarray(row_of_utt)[u], ph[s]]
    return y


def _fresh_counter(layer, value):
    layer._eps_source()
    layer._draws.fill_(value)


@pytest.mark.parametrize("period", PERIODS)
def test_bit_exact_against_composition(period):
    torch.manual_seed(100 + period)
    batch, x, off = _batch(seed=period)
    n = batch.n_utts
    layer = _layer(period, seed=period)
    rows = _rows(layer, 3 * n + 7, 0)
    y = torch.full_like(batch.wav, float("nan"))                                    # the ABI writes every sample
    assert _raw_eval(batch, layer, y) == 0                                          # no counter, no id table: d_u = u
    assert np.array_equal(y.cpu().numpy(), _expected(x, off, rows, np.arange(n)))
    for draw0, ids, n_draws in ((0, None, None), (0, np.random.default_rng(period).permutation(3 * n)[:n], 3 * n),
                                (7, None, None), (7, np.arange(n)[::-1] * 3, 3 * n)):
        _fresh_counter(layer, draw0)
        y = layer.noisy_per_utterance(batch, utt_ids=ids, n_draws=n_draws)
        want = _expected(x, off, rows, draw0 + (np.arange(n) if ids is None else ids))
        got = y.wav.cpu().numpy()
        assert np.array_equal(got, want), (draw0, ids is None)
        assert np.array_equal(got[:LEAD], x[:LEAD]) and np.array_equal(got[-TRAIL:], x[-TRAIL:])
        assert y.utt_off is batch.utt_off and y._layouts is batch._layouts
        assert int(layer._draws) == draw0 + (n if n_draws is None else n_draws)
    # external eps: (n_utts, L) rows by batch position, the counter does not move
    eps = 0.1 * torch.randn(n, period, device="cuda")
    before = int(layer._draws)
    y = layer.noisy_per_utterance(batch, external_eps=eps).wav.cpu().numpy()
    from speech_emotion_privacy_trust_b200 import cloak_ops
    rows_e, _, _ = cloak_ops.cloak_forward_raw(torch.zeros(n * period, device="cuda"), layer.locs.detach(),
                                               layer.rhos.detach(), None, eps.reshape(-1), 0, 0, 0.1, MN, MX, per_sample=True)
    rows_e = rows_e.view(n, period).cpu().numpy()                                   # the same eps through sept_cloak_fwd_f32
    assert np.array_equal(y, _expected(x, off, rows_e, np.arange(n)))
    assert int(layer._draws) == before


def _raw_eval(batch, layer, y, utt_draw=None, eps=None, x_ptr=None, y_ptr=None, ws=None):
    from speech_emotion_privacy_trust_b200 import _lib, wave_cloak
    lib = _lib.lib()
    L = layer.period
    ws = torch.empty(lib.sept_wave_cloak_eval_workspace_bytes(L) // 4 + 4, device="cuda") if ws is None else ws
    return lib.sept_wave_cloak_eval_f32(batch.wav.data_ptr() if x_ptr is None else x_ptr, batch.utt_off.data_ptr(),
                                        batch.n_utts, batch.wav.numel(), layer.locs.data_ptr(), layer.rhos.data_ptr(),
                                        None if eps is None else eps.data_ptr(), torch.initial_seed(), 0, None,
                                        None if utt_draw is None else utt_draw.data_ptr(), wave_cloak.EPS_STD,
                                        layer.min_scale, layer.max_scale, L,
                                        ws.data_ptr(), y.data_ptr() if y_ptr is None else y_ptr,
                                        torch.cuda.current_stream().cuda_stream)


def test_abi_rejects_misaligned_pointers():
    from speech_emotion_privacy_trust_b200 import _lib
    batch, _, _ = _batch()
    layer = _layer(44)
    y = torch.empty_like(batch.wav)
    ws = torch.empty(64, device="cuda")
    for kw in (dict(x_ptr=batch.wav.data_ptr() + 4), dict(y_ptr=y.data_ptr() + 8), dict(ws=ws[1:]),
               dict(eps=torch.zeros(batch.n_utts * 44 + 1, device="cuda")[1:])):
        assert _raw_eval(batch, layer, y, **kw) == _lib.SEPT_E_BADARG, kw
        assert "16-byte aligned" in _lib.lib().sept_last_error().decode()
    assert _raw_eval(batch, layer, y) == 0


def test_invariance_to_batch_position_and_sharding():
    torch.manual_seed(5)
    batch, x, off = _batch(seed=11)
    n, L = batch.n_utts, 1000
    layer = _layer(L, seed=3)
    gid = np.random.default_rng(4).permutation(50)[:n]                              # global ids of a 50-utterance corpus
    _fresh_counter(layer, 2)
    full = layer.noisy_per_utterance(batch, utt_ids=gid, n_draws=50).wav.cpu().numpy()
    from speech_emotion_privacy_trust_b200 import extraction
    for u in (6, 13, 18):                                                           # one utterance alone, same id
        alone = extraction.RaggedAudio(torch.from_numpy(x[off[u]:off[u + 1]].copy()).cuda(), np.array([0, off[u + 1] - off[u]]))
        _fresh_counter(layer, 2)
        got = layer.noisy_per_utterance(alone, utt_ids=[gid[u]], n_draws=50).wav.cpu().numpy()
        assert np.array_equal(got, full[off[u]:off[u + 1]]), u
    halves = []
    for part in (np.arange(0, n, 2), np.arange(1, n, 2)):                           # two shards, global ids
        sb = extraction.RaggedAudio.from_list([x[off[u]:off[u + 1]] for u in part])
        _fresh_counter(layer, 2)
        halves.append((part, sb.utt_off_host, layer.noisy_per_utterance(sb, utt_ids=gid[part], n_draws=50).wav.cpu().numpy()))
        assert int(layer._draws) == 52
    for part, so, y in halves:
        for i, u in enumerate(part):
            assert np.array_equal(y[so[i]:so[i + 1]], full[off[u]:off[u + 1]]), u


def test_bench_corpus_bit_exact():
    """The bench corpus (5531 utterances, 532 M samples) at L = 32 000 against the composition, built 256 utterances at a
    time on the device."""
    import bench
    from speech_emotion_privacy_trust_b200 import extraction
    torch.manual_seed(9)
    lengths = bench.corpus_lengths(bench.CORPUS_UTTS, 1234)
    off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
    batch = extraction.RaggedAudio(torch.randn(int(off[-1]), device="cuda"), off)
    L = 32000
    layer = _layer(L, seed=1)
    _fresh_counter(layer, 3)
    y = layer.noisy_per_utterance(batch).wav
    assert int(layer._draws) == 3 + len(lengths)
    for a in range(0, len(lengths), 256):
        b = min(len(lengths), a + 256)
        rows = torch.from_numpy(_rows(layer, b - a, 3 + a)).cuda().view(-1)
        s0, s1 = int(off[a]), int(off[b])
        utt = torch.repeat_interleave(torch.arange(b - a, device="cuda"), torch.from_numpy(lengths[a:b]).cuda())
        ph = torch.arange(s1 - s0, device="cuda") - torch.from_numpy(off[a:b] - s0).cuda()[utt]
        want = batch.wav[s0:s1] + rows[utt * L + ph % L]
        assert torch.equal(y[s0:s1], want), a


def test_counter_ids_and_errors():
    batch, x, off = _batch(seed=2)
    n = batch.n_utts
    layer = _layer(44)
    y0 = layer.noisy_per_utterance(batch).wav.cpu().numpy()
    y1 = layer.noisy_per_utterance(batch, n_draws=100).wav.cpu().numpy()
    assert int(layer._draws) == n + 100
    inside = order.phase_of(off, len(x), 44) >= 0
    assert not np.array_equal(y0[inside], y1[inside])                             # fresh noise on every call
    for ids, nd, msg in ((np.arange(n) - 1, None, "lie in"), (np.r_[np.arange(n - 1), 0], None, "distinct"),
                         (np.arange(n), n - 1, "lie in"), (np.arange(n + 1), None, "entries")):
        with pytest.raises(ValueError, match=msg):
            layer.noisy_per_utterance(batch, utt_ids=ids, n_draws=nd)
    with pytest.raises(ValueError, match="external_eps must be"):
        layer.noisy_per_utterance(batch, external_eps=torch.zeros(n, 40, device="cuda"))
    layer.external_eps = torch.zeros(44, device="cuda")
    with pytest.raises(ValueError, match="single sample"):
        layer.noisy_per_utterance(batch)
    assert int(layer._draws) == n + 100                                             # nothing ran


# ---- the evaluator ---------------------------------------------------------------------------------------------------
EVAL_LENGTHS = (16000, 40000, 56001, 24003, 33000, 36002)
EVAL_SPK = ["a", "b", "a", "b", "c", "c"]


def _models():
    from speech_emotion_privacy_trust_b200.dropin import baseline_models
    torch.manual_seed(21)
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0).cuda().eval()
    return mk("emotion"), mk("gender")


def _waves(lengths=EVAL_LENGTHS, seed=31):
    from speech_emotion_privacy_trust_b200 import synth
    rng = np.random.default_rng(seed)
    return [synth.speech_shaped(n, rng) for n in lengths]


def test_evaluator_against_reference_loop_per_utterance():
    from speech_emotion_privacy_trust_b200 import evaluation, extraction, normalization as nz
    base, adv = _models()
    waves = _waves()
    batch = extraction.RaggedAudio.from_list(waves)
    off = batch.utt_off_host
    layer = _layer(32000, seed=8, mn=1e-4, mx=2e-2)
    n = batch.n_utts
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False    # batch 17 vs batch 1 pick different kernels
    try:
        _fresh_counter(layer, 0)
        e_pred, g_pred, e_prob, g_prob = evaluation.wave_cloak_evaluate(layer, base, adv, batch, speaker_of_utt=EVAL_SPK,
                                                                        max_windows=7)
        assert int(layer._draws) == n
        noisy = _expected(batch.wav.cpu().numpy(), off, _rows(layer, n, 0), np.arange(n))
        feats = [extraction.logmel(extraction.RaggedAudio.from_list([noisy[off[u]:off[u + 1]]]))[0] for u in range(n)]
        feat_all = torch.cat(feats)
        fo = np.concatenate([[0], np.cumsum([f.shape[0] for f in feats])]).astype(np.int64)
        lay = extraction.Layout(fo, torch.from_numpy(fo).cuda(), torch.zeros(n + 1, dtype=torch.int32, device="cuda"))
        st = nz.speaker_stats(feat_all, lay, EVAL_SPK, whole_utterance=[True] * n)
        z = nz.normalize(feat_all, lay, st)
        for u in range(n):
            T = int(fo[u + 1] - fo[u])
            zero_row = nz.normalized_windows(feat_all, lay, st, np.array([u], np.int32), np.array([T - 1], np.int32))[0, 0, -1]
            pe, pg = [], []
            with torch.no_grad():
                for i in range(max(1, (T - 200) // 50 + 1)):
                    win = z[fo[u] + i * 50: min(fo[u + 1], fo[u] + i * 50 + 200)]
                    if win.shape[0] < 200:
                        win = torch.cat([win, zero_row.expand(200 - win.shape[0], 128)], 0)
                    pe.append(torch.softmax(base(win[None, None].contiguous()), 1)[0])
                    pg.append(torch.softmax(adv(win[None, None].contiguous()), 1)[0])
            me, mg = torch.stack(pe).mean(0).cpu().numpy(), torch.stack(pg).mean(0).cpu().numpy()
            assert np.max(np.abs(me - e_prob[u])) < 2e-4 and np.max(np.abs(mg - g_prob[u])) < 2e-4, u
            assert int(np.argmax(me)) == int(e_pred[u]) and int(np.argmax(mg)) == int(g_pred[u]), u
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def test_zero_noise_equals_clean_chain():
    from speech_emotion_privacy_trust_b200 import evaluation, extraction, normalization as nz
    from speech_emotion_privacy_trust_b200 import wave_cloak
    base, adv = _models()
    batch = extraction.RaggedAudio.from_list(_waves())
    layer = wave_cloak.WaveCloak(0.0, 0.0, period=32000).cuda()                     # mu = 0, sigma = 0
    got = evaluation.wave_cloak_evaluate(layer, base, adv, batch, speaker_of_utt=EVAL_SPK, max_windows=5)
    feat, lay = extraction.logmel(batch)
    st = nz.speaker_stats(feat, lay, EVAL_SPK, whole_utterance=[True] * batch.n_utts)
    want = evaluation._classify_windows(base, adv, lay, None, lambda a, b, wu, wt: nz.normalized_windows(feat, lay, st, wu, wt),
                                        5, feat.device)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)
    # the caller's statistics are used as given; exactly one source of statistics
    assert all(np.array_equal(g, w) for g, w in zip(evaluation.wave_cloak_evaluate(layer, base, adv, batch, stats=st,
                                                                                   max_windows=5), want))
    for kw in (dict(), dict(speaker_of_utt=EVAL_SPK, stats=st)):
        with pytest.raises(ValueError, match="exactly one"):
            evaluation.wave_cloak_evaluate(layer, base, adv, batch, **kw)


# ---- two gloo ranks on one device -------------------------------------------------------------------------------
DP_LENGTHS = (16000, 40000, 56001, 24003, 33000, 47005, 20000, 36002, 52003)
DP_SPK = ["a", "b", "a", "b", "a", "c", "c", "b", "a"]


def _dp_eval(mine, n_all, stats_fn):
    """(noisy audio per utterance, probabilities) of the utterances `mine` with global ids: the layer's counter at 0,
    noisy_per_utterance, then wave_cloak_evaluate on the same utterances (the counter then at n_all)."""
    from speech_emotion_privacy_trust_b200 import evaluation, extraction
    base, adv = _models()
    waves = _waves(DP_LENGTHS, seed=41)
    torch.manual_seed(0)
    layer = _layer(32000, seed=12, mn=1e-4, mx=2e-2)
    batch = extraction.RaggedAudio.from_list([waves[u] for u in mine])
    noisy = layer.noisy_per_utterance(batch, utt_ids=mine, n_draws=n_all)                      # draws 0 .. n_all - 1
    feat, lay = extraction.logmel(layer.noisy_per_utterance(batch, utt_ids=mine, n_draws=n_all))   # n_all .. 2 n_all - 1
    st = stats_fn(feat, lay, [DP_SPK[u] for u in mine])
    _fresh_counter(layer, n_all)                                    # the evaluator draws what the statistics were built on
    res = evaluation.wave_cloak_evaluate(layer, base, adv, batch, stats=st, utt_ids=mine, n_draws=n_all)
    y, so = noisy.wav.cpu().numpy(), noisy.utt_off_host
    return [y[so[i]:so[i + 1]] for i in range(len(mine))], res


def _dp_worker(rank, world, init_file, out_dir):
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=f"file://{init_file}", rank=rank, world_size=world,
                            timeout=timedelta(seconds=120))
    try:
        from speech_emotion_privacy_trust_b200 import normalization as nz, parallel
        mine = parallel.shard_by_length(DP_LENGTHS, world)[rank]
        whole = lambda f, lay, s: nz.speaker_stats_distributed(f, lay, s, ["a", "b", "c"], whole_utterance=[True] * len(s))
        audio, res = _dp_eval(mine, len(DP_LENGTHS), whole)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), mine=mine, e_prob=res[2], g_prob=res[3], e_pred=res[0],
                 g_pred=res[1], **{f"a{u}": a for u, a in zip(mine, audio)})
    finally:
        dist.destroy_process_group()


def test_two_gloo_ranks_match_one_gpu(tmp_path):
    from speech_emotion_privacy_trust_b200 import normalization as nz
    mp.spawn(_dp_worker, args=(2, str(tmp_path / "store"), str(tmp_path)), nprocs=2, join=True)
    allu = list(range(len(DP_LENGTHS)))
    audio, (e_pred, g_pred, e_prob, g_prob) = _dp_eval(
        allu, len(DP_LENGTHS), lambda f, lay, s: nz.speaker_stats(f, lay, s, whole_utterance=[True] * len(s)))
    seen = set()
    for r in range(2):
        res = np.load(tmp_path / f"r{r}.npz")
        for i, u in enumerate(res["mine"]):
            u = int(u)
            seen.add(u)
            assert np.array_equal(res[f"a{u}"], audio[u]), u                       # the same noisy audio, bit for bit
            assert np.max(np.abs(res["e_prob"][i] - e_prob[u])) < 1e-4 and np.max(np.abs(res["g_prob"][i] - g_prob[u])) < 1e-4
            assert res["e_pred"][i] == e_pred[u] and res["g_pred"][i] == g_pred[u]
    assert seen == set(allu)
