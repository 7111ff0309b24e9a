"""GPU parity of the fused cloak / gradient-reversal kernels against the golden vectors of the real reference modules
(eps supplied externally; north_star tolerance 1e-6) and of the drop-in modules against a plain PyTorch fp32
composition of the same ops."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 1e-6


@pytest.fixture(scope="module")
def mods():
    from speech_emotion_privacy_trust_b200 import dropin
    dropin.install()
    import baseline_models
    import cloak_models
    import reversal_gradient
    return cloak_models, reversal_gradient, baseline_models


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("tag", ["nomask", "mask"])
def test_cloak_layer_golden_forward_backward(mods, golden_cloak, tag):
    cloak_models, reversal_gradient, _ = mods
    g = golden_cloak
    mn, mx, lam = float(g["min_scale"]), float(g["max_scale"]), float(g["lambda"])
    layer = cloak_models.cloak_noise(_t(g[f"{tag}_locs"]).cpu(), torch.ones(g[f"{tag}_locs"].shape), mn, mx, "cuda").cuda()
    with torch.no_grad():
        layer.rhos.copy_(_t(g[f"{tag}_rhos"]))
    layer.external_eps = _t(g[f"{tag}_eps"])
    mask = _t(g["mask_mask"]) if tag == "mask" else None
    x = _t(g[f"{tag}_x"]).requires_grad_(True)
    assert float((layer.scales() - _t(g[f"{tag}_sigma"])).abs().max()) < TOL
    # (a) the reference's own composition: cloak layer, then a separate GradientReversal on one branch
    y = layer(x, mask) if mask is not None else layer(x)
    assert float((y - _t(g[f"{tag}_out"])).abs().max()) < TOL
    y_rev = reversal_gradient.GradientReversalFunction.apply(y, lam)
    ((y * _t(g[f"{tag}_g_a"])).sum() + (y_rev * _t(g[f"{tag}_g_b"])).sum()).backward()
    for got, key in ((layer.locs.grad, "dlocs"), (layer.rhos.grad, "drhos"), (x.grad, "dx")):
        scale = max(1.0, float(np.abs(g[f"{tag}_{key}"]).max()))
        assert float((got - _t(g[f"{tag}_{key}"])).abs().max()) < TOL * scale * 4, key
    # (b) the fused twin: one backward kernel takes both upstream gradients and applies -lambda itself
    layer.zero_grad()
    x2 = _t(g[f"{tag}_x"]).requires_grad_(True)
    ya, yb = layer.forward_with_reversed_twin(x2, mask, lam)
    assert torch.equal(ya, y.detach()) and ya.data_ptr() == yb.data_ptr()
    ((ya * _t(g[f"{tag}_g_a"])).sum() + (yb * _t(g[f"{tag}_g_b"])).sum()).backward()
    for got, key in ((layer.locs.grad, "dlocs"), (layer.rhos.grad, "drhos"), (x2.grad, "dx")):
        scale = max(1.0, float(np.abs(g[f"{tag}_{key}"]).max()))
        assert float((got - _t(g[f"{tag}_{key}"])).abs().max()) < TOL * scale * 4, key


def test_gradient_reversal_golden(mods, golden_cloak):
    _, reversal_gradient, _ = mods
    g = golden_cloak
    z = _t(g["grl_g"] * 0 + 1.0).requires_grad_(True)
    out = reversal_gradient.GradientReversal(float(g["grl_lambda"]))(z)
    assert torch.equal(out, z)
    out.backward(_t(g["grl_g"]))
    assert np.array_equal(z.grad.cpu().numpy(), g["grl_dx"])      # bit exact: one fp32 multiply
    assert reversal_gradient.ReverseLayerF is reversal_gradient.GradientReversalFunction


def test_cloak_full_size_vs_torch_fp32(mods):
    """B=64, W=200, F=128 (config 2) against the same formula written with torch ops in fp32 on the GPU."""
    cloak_models, _, _ = mods
    torch.manual_seed(3)
    B, W, F = 64, 200, 128
    layer = cloak_models.cloak_noise(0.1 * torch.randn(1, W, F), torch.ones(1, W, F), 0.01, 5.0, "cuda").cuda()
    with torch.no_grad():
        layer.rhos.add_(torch.randn(1, W, F, device="cuda"))
    eps = 0.1 * torch.randn(1, W, F, device="cuda")
    layer.external_eps = eps
    mask = (torch.rand(1, W, F, device="cuda") > 0.4).float()
    x = torch.randn(B, 1, W, F, device="cuda", requires_grad=True)
    ga, gb, lam = torch.randn(B, 1, W, F, device="cuda"), torch.randn(B, 1, W, F, device="cuda"), 0.1
    ya, yb = layer.forward_with_reversed_twin(x, mask, lam)
    ((ya * ga).sum() + (yb * gb).sum()).backward()
    got = (ya.detach().clone(), layer.locs.grad.clone(), layer.rhos.grad.clone(), x.grad.clone())
    layer.zero_grad()
    xr = x.detach().clone().requires_grad_(True)
    ref_y = xr * mask + (layer.locs + layer.scales() * (eps * mask))
    gtot = ga - lam * gb
    (ref_y * gtot).sum().backward()
    assert float((got[0] - ref_y.detach()).abs().max()) < TOL
    assert float((got[3] - xr.grad).abs().max()) < TOL
    # batch reductions of 64 O(1) terms: compare to an fp64 sum, allow a few fp32 ulps of the sum's magnitude
    d64 = gtot.double().sum(0)
    assert float((got[1].double() - d64).abs().max()) < 2e-5
    assert float((got[1] - layer.locs.grad).abs().max()) < 2e-5
    assert float((got[2] - layer.rhos.grad).abs().max()) < 2e-5 * max(1.0, float(layer.rhos.grad.abs().max()))
    # deterministic reduction
    layer.zero_grad()
    ya, yb = layer.forward_with_reversed_twin(x, mask, lam)
    ((ya * ga).sum() + (yb * gb).sum()).backward()
    assert torch.equal(layer.locs.grad, got[1]) and torch.equal(layer.rhos.grad, got[2])


def test_device_philox_noise(mods):
    cloak_models, _, _ = mods
    torch.manual_seed(8)
    layer = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cuda").cuda()
    x = torch.zeros(4, 1, 200, 128, device="cuda")
    sig = layer.scales().detach()
    e1 = (layer(x)[0] / sig)                                   # locs = 0 -> y = sigma * eps
    e2 = (layer(x)[0] / sig)
    assert abs(float(e1.mean())) < 2e-3 and abs(float(e1.std()) - 0.1) < 2e-3      # N(0, 0.1), 25 600 samples
    assert not torch.equal(e1, e2)                              # a fresh sample per forward ...
    y = layer(x)
    assert torch.equal(y[0], y[3])                              # ... shared by the whole batch (cloak_models.py:47)
    torch.manual_seed(8)
    again = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cuda").cuda()
    assert torch.equal(again(x)[0] / sig, e1)                   # same seed, same draw index -> same eps on every rank
    n = layer.sample_noise()
    assert n.shape == (1, 200, 128) and n.requires_grad
    k = float(((e1.flatten() / 0.1) ** 4).mean())
    assert 2.7 < k < 3.3                                        # Gaussian kurtosis


def test_grl_model_matches_unfused_composition(mods):
    """two_d_cnn_lstm_syn_with_grl: the fused twin path against the reference's literal composition (cloak layer ->
    GradientReversal module -> gender conv), same weights, dropout off, eps shared."""
    cloak_models, reversal_gradient, baseline_models = mods
    torch.manual_seed(5)
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0)
    noise = cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cuda")
    model = cloak_models.two_d_cnn_lstm_syn_with_grl(mk("emotion"), mk("gender"), noise, 0.1).cuda().train()
    for mod in model.modules():
        if isinstance(mod, (torch.nn.Dropout, torch.nn.Dropout2d)):
            mod.p = 0.0
        if isinstance(mod, torch.nn.GRU):
            mod.dropout = 0.0
        if isinstance(mod, torch.nn.BatchNorm2d):
            mod.eval()
    eps = 0.1 * torch.randn(1, 200, 128, device="cuda")
    model.intermed.external_eps = eps
    x = torch.randn(8, 1, 200, 128, device="cuda")
    emo, gen = torch.randint(0, 4, (8,), device="cuda"), torch.randint(0, 2, (8,), device="cuda")
    ce = torch.nn.functional.cross_entropy

    def grads(fused):
        model.zero_grad()
        if fused:
            p1, p2, noisy = model(x, pooling="mean")
        else:
            y = model.intermed(x)
            noisy = y.detach()
            z1 = baseline_models.sequence_features(model.original_model, y).mean(dim=1)
            p1 = baseline_models.classify(model.original_model, z1, None, pred="emotion")
            z2 = baseline_models.sequence_features(model.gender_model, y).mean(dim=1)     # conv = Sequential(GRL, conv)
            p2 = baseline_models.classify(model.gender_model, z2, None, pred="gender")
        (ce(p1, emo) + 0.1 * ce(p2, gen)).backward()
        conv_w = model.gender_model.conv[1][0].weight.grad.clone()
        return p1.detach(), p2.detach(), noisy, model.intermed.locs.grad.clone(), model.intermed.rhos.grad.clone(), conv_w

    a, b = grads(True), grads(False)
    assert a[0].shape == (8, 4) and a[1].shape == (8, 2) and a[2].shape == (8, 1, 200, 128)
    assert torch.equal(a[2], b[2])
    for i, name in ((0, "preds1"), (1, "preds2"), (3, "dlocs"), (4, "drhos"), (5, "gender conv wgrad")):
        scale = max(1e-3, float(b[i].abs().max()))
        assert float((a[i] - b[i]).abs().max()) < 2e-3 * scale, name     # cuDNN conv/GRU (TF32-capable) sit in between
    assert all(p.grad is None for p in model.original_model.parameters())


def test_cloak_inside_cuda_graph_draws_fresh_noise(mods):
    """The Philox draw counter lives on the device: replaying a captured forward yields a new eps each time, and the
    sequence equals the eager one for the same seed (what keeps data-parallel ranks in step)."""
    cloak_models, _, _ = mods
    x = torch.zeros(2, 1, 200, 128, device="cuda")

    def fresh():
        torch.manual_seed(11)
        return cloak_models.cloak_noise(torch.zeros(1, 200, 128), torch.ones(1, 200, 128), 0.01, 10.0, "cuda").cuda()
    eager = fresh()
    want = [eager(x).clone() for _ in range(4)]
    layer = fresh()
    with torch.no_grad():
        first = layer(x).clone()                          # warm-up (allocations) consumes draw 0
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            y = layer(x)
        outs = []
        for _ in range(3):
            g.replay()
            outs.append(y.clone())
    assert torch.equal(first, want[0])
    # capture itself does not execute kernels, so the replays are draws 1, 2, 3
    for got, ref in zip(outs, want[1:]):
        assert torch.equal(got, ref)
    assert not torch.equal(outs[0], outs[1])


def test_distributed_speaker_stats_single_rank_equals_local():
    from speech_emotion_privacy_trust_b200 import normalization as nz
    from speech_emotion_privacy_trust_b200.extraction import Layout
    rng = np.random.default_rng(3)
    frames = [230, 410, 199, 305]
    spk = ["x", "y", "x", "z"]
    feats = [(rng.standard_normal((T, 128)) * 4 - 20).astype(np.float32) for T in frames]
    fo = np.concatenate([[0], np.cumsum(frames)]).astype(np.int64)
    lay = Layout(fo, torch.from_numpy(fo).cuda(), torch.zeros(len(fo), dtype=torch.int32, device="cuda"))
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    a = nz.speaker_stats(feat, lay, spk)
    b = nz.speaker_stats_distributed(feat, lay, spk, all_speakers=["z", "y", "x", "absent"])
    da, db = a.as_dict(), b.as_dict()
    for s in ("x", "y", "z"):
        for k in ("count", "mean", "std", "min", "max"):
            assert np.allclose(da[s][k], db[s][k], rtol=0, atol=2e-5), (s, k)
    for k, want in (("count", 0.0), ("mean", 0.0), ("std", 0.0), ("min", np.inf), ("max", -np.inf)):
        assert np.all(db["absent"][k] == want), (k, db["absent"][k])       # in every feature of the row no rank holds
    za, zb = nz.normalize(feat, lay, a), nz.normalize(feat, lay, b)
    assert float((za - zb).abs().max()) < 1e-4


def test_batched_evaluation_equals_reference_window_loop(mods):
    """evaluation.cloak_evaluate (all windows in one forward, per-window eps) against the reference's literal loop
    (adversary_cloak_evaluation.py:60-93): one window at a time through the cloak layer with the same eps."""
    cloak_models, _, baseline_models = mods
    from speech_emotion_privacy_trust_b200 import evaluation, normalization as nz
    from speech_emotion_privacy_trust_b200.extraction import Layout
    torch.manual_seed(21)
    rng = np.random.default_rng(21)
    frames = [431, 150, 260, 777]
    spk = ["a", "b", "a", "b"]
    feats = [(rng.standard_normal((T, 128)) * 6 - 35).astype(np.float32) for T in frames]
    fo = np.concatenate([[0], np.cumsum(frames)]).astype(np.int64)
    lay = Layout(fo, torch.from_numpy(fo).cuda(), torch.zeros(len(fo), dtype=torch.int32, device="cuda"))
    feat = torch.from_numpy(np.concatenate(feats)).cuda()
    st = nz.speaker_stats(feat, lay, spk, whole_utterance=[True] * 4)
    mk = lambda pred: baseline_models.two_d_cnn_lstm(1, 128, 5, lstm_hidden_size=64, pred=pred, global_feature=0).cuda().eval()
    base, adv = mk("emotion"), mk("gender")
    layer = cloak_models.cloak_noise(0.05 * torch.randn(1, 200, 128), torch.ones(1, 200, 128), 0.01, 5.0, "cuda").cuda()
    with torch.no_grad():
        layer.rhos.add_(torch.randn(1, 200, 128, device="cuda"))
    mask = evaluation.suppression_mask(layer, 40)
    sig = layer.scales().detach()
    assert abs(float((mask == 0).float().mean()) - 0.6) < 0.01            # the 60 % largest sigmas are suppressed
    wu, wt = evaluation.eval_window_table(lay)
    assert [int((wu == u).sum()) for u in range(4)] == [(431 - 200) // 50 + 1, 1, 2, (777 - 200) // 50 + 1]
    eps = 0.1 * torch.randn(len(wu), 200, 128, device="cuda")
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False    # batch 17 vs batch 1 pick different kernels
    e_pred, g_pred, e_prob, g_prob = evaluation.cloak_evaluate(layer, base, adv, feat, lay, st, mask=mask, external_eps=eps)
    from speech_emotion_privacy_trust_b200 import cloak_ops
    xw = nz.normalized_windows(feat, lay, st, wu, wt)
    noisy_all, _, _ = cloak_ops.cloak_forward_raw(xw, layer.locs.detach().contiguous(), layer.rhos.detach().contiguous(), mask.contiguous(),
                                                  eps.reshape(-1), 0, 0, 0.1, 0.01, 5.0, per_sample=True)
    # the reference loop
    z = nz.normalize(feat, lay, st)
    zero_row = nz.normalized_windows(feat, lay, st, np.array([1], np.int32), np.array([0], np.int32))[0, 0, -1]   # padded row of utt 1
    w = 0
    for u, T in enumerate(frames):
        pe, pg = [], []
        for i in range(max(1, (T - 200) // 50 + 1)):
            win = z[fo[u] + i * 50: min(fo[u + 1], fo[u] + i * 50 + 200)]
            if win.shape[0] < 200:
                win = torch.cat([win, zero_row.expand(200 - win.shape[0], 128)], 0)
            layer.external_eps = eps[w:w + 1]
            with torch.no_grad():
                noisy = layer(win[None, None].contiguous(), mask)
                assert torch.equal(noisy[0], noisy_all[w])              # the per-window eps path is bit identical
                pe.append(torch.softmax(base(noisy), 1)[0])
                pg.append(torch.softmax(adv(noisy), 1)[0])
            w += 1
        me, mg = torch.stack(pe).mean(0).cpu().numpy(), torch.stack(pg).mean(0).cpu().numpy()
        assert np.max(np.abs(me - e_prob[u])) < 2e-4 and np.max(np.abs(mg - g_prob[u])) < 2e-4
        assert int(np.argmax(me)) == int(e_pred[u]) and int(np.argmax(mg)) == int(g_pred[u])
    layer.external_eps = None
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    # device-drawn noise: per-window samples differ, and the draw counter advanced by the number of windows
    before = int(layer._eps_source()[2].item()) if layer._draws is not None else 0
    evaluation.cloak_evaluate(layer, base, adv, feat, lay, st, mask=None)
    assert int(layer._draws.item()) - before == len(wu)
