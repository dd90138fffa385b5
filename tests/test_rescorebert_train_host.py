"""RescoreBert distillation without a GPU: the closed-form MD / MWER gradients the device's loss
kernel evaluates (include/pllb.h) against torch autograd, the batching of RescoreBert/train.py, and
the trainer failing loudly when no B200 is visible."""
import numpy as np
import pytest
import torch

from asr_rescoring_b200 import _lib, synth
from asr_rescoring_b200.RescoreBert import train as rb_train
from oracle import rescorebert_train_oracle as rto


def _autograd_dscore(s, target, am, err, group, **w):
    st = torch.tensor(s, dtype=torch.float64, requires_grad=True)
    loss, _, _ = rto.losses(st, target, am, err, group, **w)
    loss.backward()
    return float(loss.detach()), st.grad.numpy()


@pytest.mark.parametrize("weights", [dict(md_weight=1.0, mwer_weight=0.0, am_weight=1.0),
                                     dict(md_weight=1.0, mwer_weight=1.0, am_weight=1.0),
                                     dict(md_weight=0.3, mwer_weight=2.0, am_weight=0.7),
                                     dict(md_weight=0.0, mwer_weight=1.0, am_weight=0.0)])
def test_closed_form_gradients_match_autograd(weights):
    rng = np.random.default_rng(3)
    sizes = [10, 1, 4, 7, 3, 10]                    # a group of one hypothesis, too
    group = np.repeat(np.arange(len(sizes)), sizes)
    B = len(group)
    s = rng.normal(0, 2, B)
    target = rng.normal(-30, 8, B)
    am = rng.normal(-3, 2, B)
    err = rng.integers(0, 4, B) / 10.0
    s[3] = s[4]; am[3] = am[4]                      # a tie inside a group
    err[10:11] = 0.25
    err[11:15] = 0.5                                # a group whose errors are all equal
    loss, auto = _autograd_dscore(s, target, am, err, group, **weights)
    closed = rto.closed_form_dscore(s, target, am, err, group, **weights)
    assert np.allclose(closed, auto, rtol=1e-10, atol=1e-13)
    assert np.isfinite(loss)
    if weights["mwer_weight"] > 0:
        # equal errors: no MWER gradient in that group; a group of one: P = 1, no contribution
        md_only = rto.closed_form_dscore(s, target, am, err, group, md_weight=weights["md_weight"])
        assert np.allclose(closed[10:15], md_only[10:15], atol=1e-15)


def test_mwer_loss_of_a_singleton_group_is_zero():
    s, t, a = np.array([0.5]), np.array([0.5]), np.array([-1.0])
    total, md, mwer = rto.losses(torch.tensor(s), t, a, np.array([0.3]), np.array([0]), mwer_weight=1.0)
    assert float(total) == 0.0 and float(mwer) == 0.0


def test_make_batches_groups_padding_and_lengths():
    tokens = {"u1": {"hyp_1": [5, 6, 7], "hyp_2": [5, 6]}, "u2": {"hyp_1": [9]}, "u3": {"hyp_1": [], "hyp_2": [4, 4, 4, 4]}}
    val = lambda k: {u: {h: float(k * 10 + i) for i, h in enumerate(hs)} for u, hs in tokens.items()}   # noqa: E731
    pll, am, cer = val(1), val(2), val(3)
    batches = rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=2)
    assert len(batches) == 2
    b0, b1 = batches
    assert b0["keys"] == [("u1", "hyp_1"), ("u1", "hyp_2"), ("u2", "hyp_1")]
    assert b0["group"].tolist() == [0, 0, 1] and b1["group"].tolist() == [0, 0]
    assert b0["input_ids"].tolist() == [[101, 5, 6, 7, 102], [101, 5, 6, 102, 0], [101, 9, 102, 0, 0]]
    assert b0["attention_mask"].sum(1).tolist() == [5, 4, 3] and b0["input_ids"].dtype == np.int32
    assert b1["input_ids"].tolist() == [[101, 102, 0, 0, 0, 0], [101, 4, 4, 4, 4, 102]]
    assert b0["target"].tolist() == [10.0, 11.0, 10.0] and b0["am"].tolist() == [20.0, 21.0, 20.0]
    assert b1["err"].tolist() == [30.0, 31.0] and b1["err"].dtype == np.float32
    assert rb_train.batch_capacity(batches) == (15, 6)
    with pytest.raises(ValueError):
        rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=0)


@pytest.mark.skipif(_lib.load().pllb_device_count() > 0, reason="a GPU is present")
def test_cls_trainer_fails_loudly_without_gpu():
    from asr_rescoring_b200 import engine
    sd = synth.random_rescorebert_state_dict(synth.BERT_TINY, 1)
    with pytest.raises(_lib.PllbError):
        engine.ClsTrainer(sd, synth.BERT_TINY)
    with pytest.raises(ValueError):                  # not a RescoreBert checkpoint: checked before the device
        engine.ClsTrainer({k: v for k, v in sd.items() if not k.startswith("linear.")}, synth.BERT_TINY)
