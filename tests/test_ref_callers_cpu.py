"""The reference's caller scripts (verbatim copies under tests/ref_fixture/) against the drop-in modules, CPU part:
their import lines resolve, the harness drives the reference's own train()/test() end to end with the reference's
models, and the drop-ins refuse to compute without a CUDA device (no CPU fallback)."""
import hashlib
import importlib.util
import json

import numpy as np
import pytest
import torch

import ref_harness as H

SCRIPTS = ["training_cloak_with_grl", "training_cloak", "adversary_cloak_evaluation", "training_adversary_baselines"]


def test_vendored_fixture_equals_the_reference():
    """Every vendored file still has the SHA-256 that vendor.py recorded from the reference when it copied it."""
    spec = importlib.util.spec_from_file_location("ref_fixture_vendor", H.FIXTURE / "vendor.py")
    vendor = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(vendor)
    want = json.loads(vendor.DIGESTS.read_text())
    assert sorted(want) == sorted(vendor.FILES)
    got = {rel: hashlib.sha256((H.FIXTURE / rel).read_bytes()).hexdigest() for rel in vendor.FILES}
    assert got == want


@pytest.mark.parametrize("script", SCRIPTS)
def test_driver_import_lines_resolve_to_the_dropins(script):
    """ADVICE r1 (high): every `from baseline_models import ...` / `from cloak_models import ...` line of the four
    training scripts must work after dropin.install() -- executed here by importing the unmodified scripts."""
    mod = H.load_driver(script, "dropin")
    dropin_dir = H.REPO / "speech_emotion_privacy_trust_b200" / "dropin"
    assert mod.flat_origins["baseline_models"] == dropin_dir
    assert mod.flat_origins["training_tools"] == H.FIXTURE / "utils"          # utilities stay the reference's
    if script != "training_adversary_baselines":
        assert mod.flat_origins["cloak_models"] == dropin_dir and mod.flat_origins["reversal_gradient"] == dropin_dir
    ref = H.load_driver(script, "reference")
    assert ref.flat_origins["baseline_models"] == H.FIXTURE / "model"
    assert ref.two_d_cnn_lstm is not mod.two_d_cnn_lstm


def test_added_baseline_classes_keep_reference_keys_and_forward():
    """one_d_cnn_lstm / deep_two_d_cnn_lstm_tmp / two_d_cnn: state_dicts interchangeable with the reference classes,
    same eval-mode outputs from the same weights; two_d_cnn's forward raises in both (channel mismatch, :548/:552)."""
    ref = H.load_driver("training_adversary_baselines", "reference")
    new = H.load_driver("training_adversary_baselines", "dropin")
    torch.manual_seed(0)
    x = torch.randn(2, 1, 200, 128)
    cases = [("one_d_cnn_lstm", dict(lstm_hidden_size=64, global_feature=0), True),
             ("one_d_cnn_lstm", dict(lstm_hidden_size=256, global_feature=0, att="self_att"), False),     # 512*4 != 512: raises
             ("deep_two_d_cnn_lstm_tmp", dict(lstm_hidden_size=32, global_feature=0), True),
             ("deep_two_d_cnn_lstm_tmp", dict(lstm_hidden_size=32, global_feature=0, rnn_cell="gru", att="self_att"), False)]
    for name, kw, runs in cases:
        a = getattr(ref, name)(1, 128, 64, **kw).eval()
        b = getattr(new, name)(1, 128, 64, **kw).eval()
        assert {k: tuple(v.shape) for k, v in a.state_dict().items()} == {k: tuple(v.shape) for k, v in b.state_dict().items()}
        assert list(a.state_dict()) == list(b.state_dict())
        b.load_state_dict(a.state_dict(), strict=True)
        outs = []
        for m in (a, b):
            try:
                with torch.no_grad():
                    outs.append(m(x))
            except RuntimeError as e:
                outs.append(type(e))
        if runs:
            assert torch.equal(outs[0], outs[1]), name
        else:
            assert outs[0] is outs[1] or (torch.is_tensor(outs[0]) and torch.equal(outs[0], outs[1])), name
    a, b = ref.two_d_cnn(1, 128, 64, global_feature=0), new.two_d_cnn(1, 128, 64, global_feature=0)
    assert list(a.state_dict()) == list(b.state_dict())
    assert all(a.state_dict()[k].shape == b.state_dict()[k].shape for k in a.state_dict())
    for m in (a, b):
        with pytest.raises(RuntimeError):
            m(x)


def test_reference_train_and_test_run_under_the_harness_on_cpu():
    """Harness self-check with the reference's own models: train()/test() of training_cloak_with_grl.py and
    training_cloak.py run unmodified, eps comes from the tape once per forward, losses are finite, sigma moved."""
    torch.set_num_threads(min(8, torch.get_num_threads()))
    tr, va, te = H.synthetic_split(16, 1), H.synthetic_split(8, 2), H.synthetic_split(3, 3, frames=(200, 310))
    mod = H.load_driver("training_cloak_with_grl", "reference")
    torch.manual_seed(8)
    rec = []
    res, model, tape = H.run_grl_training(mod, "cpu", tr, va, te, epochs=1, batch_size=8, record=rec)
    n_test_windows = sum((d["data"].shape[1] - 200) // 50 + 1 for d in te.values())
    assert tape.draws == 2 + 1 + n_test_windows and len(rec) == 2
    assert rec[0][0].shape == (8, 4) and rec[0][1].shape == (8, 2)
    r = res[0]
    assert np.isfinite(r["train"]["combine"]["loss"]["emotion"]) and np.isfinite(r["validate"]["combine"]["loss"]["emotion"])
    assert 0.0 <= r["test"]["combine"]["rec"]["emotion"] <= 1.0
    assert float((model.intermed.rhos.detach() + 2).abs().max()) > 0 and float(model.intermed.locs.detach().abs().max()) > 0
    assert all(not p.requires_grad for p in model.original_model.parameters())

    mod2 = H.load_driver("training_cloak", "reference")
    res2, model2, tape2 = H.run_cloak_training(mod2, "cpu", tr, va, te, epochs=1, batch_size=8)
    assert np.isfinite(res2[0]["train"]["combine"]["loss"]["emotion"]) and tape2.draws == 3 + n_test_windows


def test_dropins_refuse_to_compute_on_cpu():
    """No CPU fallback: the same harness with the drop-ins on a CPU device fails loudly instead of computing."""
    tr, va, te = H.synthetic_split(8, 1), H.synthetic_split(8, 2), H.synthetic_split(3, 3)
    mod = H.load_driver("training_cloak_with_grl", "dropin")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        H.run_grl_training(mod, "cpu", tr, va, te, epochs=1, batch_size=8)
