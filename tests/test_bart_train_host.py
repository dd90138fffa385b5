"""Host side of CorrectBart fine-tuning (DESIGN.md §3.13): struct layouts, the decoder-input rule, batch
building, the Python-side rejections and the fp32 oracle (oracle/bart_train_oracle.py) against transformers."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from asr_rescoring_b200 import _lib, engine  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402
from oracle import bart_train_oracle as bto  # noqa: E402


def _header_fields(name):
    src = open(os.path.join(ROOT, "include", "pllb.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    out = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            out += [n.strip().lstrip("*") for n in decl.split(None, 1)[1].split(",")]
    return out


def test_train_desc_layout_matches_header():
    assert [f for f, _ in _lib.S2sTrainDesc._fields_] == _header_fields("pllb_s2s_train_desc")
    assert ctypes.sizeof(_lib.S2sTrainDesc) == 64
    assert _lib.S2sTrainDesc.seed.offset == 32


def test_signatures_declared():
    src = open(os.path.join(ROOT, "include", "pllb.h")).read()
    for name in ("pllb_s2s_train_create", "pllb_s2s_train_step_host", "pllb_s2s_train_export",
                 "pllb_s2s_train_export_grads"):
        assert name in _lib.SIGNATURES and re.search(r"\b%s\(" % name, src)


@pytest.mark.parametrize("label_pad", [-100, 0])
def test_decoder_input_equals_shift_tokens_right(label_pad):
    import torch
    from transformers.models.bart.modeling_bart import shift_tokens_right
    rng = np.random.default_rng(0)
    lab = rng.integers(5, 300, (4, 7))
    lab[1, 4:] = label_pad
    lab[3, 2:] = label_pad
    exp = shift_tokens_right(torch.tensor(lab), 0, 102).numpy()
    assert np.array_equal(engine.shift_tokens_right(lab, 0, 102), exp)


class _Tok:
    def encode(self, text):
        return [200 + ord(c) - ord("a") for c in text]


def test_make_batches_and_pairs():
    from asr_rescoring_b200.CorrectBart.train import batch_capacity, make_batches, one_hyp_pairs
    hyps, refs = one_hyp_pairs({"u1": {"hyp_1": "ab", "hyp_2": "x"}, "u2": {"hyp_1": "abcd"}}, {"u2": "abc", "u1": "b"})
    assert hyps == ["ab", "abcd"] and refs == ["b", "abc"]
    with pytest.raises(ValueError):
        one_hyp_pairs({"u1": {"hyp_1": "a"}}, {})
    b = make_batches(_Tok(), hyps, refs, 8)
    assert len(b) == 1
    assert b[0]["input_ids"].tolist() == [[101, 200, 201, 102, 0, 0], [101, 200, 201, 202, 203, 102]]
    assert b[0]["attention_mask"].tolist() == [[1, 1, 1, 1, 0, 0], [1] * 6]
    assert b[0]["labels"].tolist() == [[101, 201, 102, -100, -100], [101, 200, 201, 202, 102]]
    assert make_batches(_Tok(), hyps, refs, 8, label_pad=0)[0]["labels"][0].tolist() == [101, 201, 102, 0, 0]
    assert [x["input_ids"].shape[0] for x in make_batches(_Tok(), hyps * 3, refs * 3, 4)] == [4, 2]
    assert batch_capacity(b) == (2, 6, 5)
    with pytest.raises(ValueError):
        make_batches(_Tok(), hyps, refs, 0)
    with pytest.raises(ValueError):
        make_batches(_Tok(), hyps, refs[:1], 2)


def test_python_rejections():
    cfg = bo.bart_config(d_model=256, layers=1, ffn=512, vocab=300, max_position=32)
    sd = bo.make_model(cfg).state_dict()
    d = cfg.to_dict()
    with pytest.raises(ValueError, match="activation_dropout"):
        engine.Seq2SeqTrainer(sd, dict(d, activation_dropout=0.1))
    with pytest.raises(ValueError, match="bf16"):
        engine.Seq2SeqTrainer(sd, d, operand_dtype="fp16")
    with pytest.raises(ValueError):
        engine.Seq2SeqTrainer(sd, dict(d, activation_function="relu"))
    with pytest.raises(ValueError, match="model.shared.weight"):     # the table only under a tied alias
        engine.Seq2SeqTrainer({("model.encoder.embed_tokens.weight" if k == "model.shared.weight" else k): v
                               for k, v in sd.items() if k != "model.encoder.embed_tokens.weight"}, d)
    with pytest.raises(ValueError, match="prefix"):
        engine._prefix_lengths(np.array([[1, 0, 1]]), (1, 3))


def _tiny():
    cfg = bo.bart_config(d_model=128, layers=1, ffn=256, vocab=120, max_position=32, scale_embedding=True)
    cfg.encoder_attention_heads = cfg.decoder_attention_heads = 2
    return cfg, bo.make_model(cfg, seed=1)


def _batch():
    ids = np.array([[101, 20, 30, 102, 0], [101, 40, 50, 60, 102]])
    mask = (np.arange(5)[None] < np.array([[4], [5]])).astype(np.int64)
    labels = np.array([[101, 21, 102, -100], [101, 41, 51, 102]])
    return ids, mask, labels


def test_oracle_loss_equals_forward_and_token_mean():
    import copy
    import torch
    cfg, m = _tiny()
    ids, mask, labels = _batch()
    with torch.no_grad():
        ref = copy.deepcopy(m).train()
        exp = float(ref(input_ids=torch.tensor(ids), attention_mask=torch.tensor(mask), labels=torch.tensor(labels)).loss)
    loss, tl, grads, _ = bto.step(m, ids, mask, labels, update=False)
    assert loss == pytest.approx(exp, rel=1e-6)
    assert np.all(tl[labels == -100] == 0)
    assert tl[labels != -100].mean() == pytest.approx(loss, rel=1e-5)
    assert "model.shared.weight" in grads and "lm_head.weight" not in grads      # tied: once
    assert float(grads["model.encoder.embed_positions.weight"][:2].abs().max()) == 0.0


def test_oracle_adamw_keeps_bias_and_decays_position_rows():
    cfg, m = _tiny()
    before = {k: v.clone() for k, v in m.state_dict().items()}
    ids, mask, labels = _batch()
    lr, wd = 1e-3, 0.01
    bto.step(m, ids, mask, labels, lr=lr, weight_decay=wd)
    after = m.state_dict()
    assert np.array_equal(after["final_logits_bias"].numpy(), before["final_logits_bias"].numpy())
    for k in ("model.encoder.embed_positions.weight", "model.decoder.embed_positions.weight"):
        np.testing.assert_allclose(after[k][:2].numpy(), before[k][:2].numpy() * (1 - lr * wd), rtol=1e-6)
    assert not np.array_equal(after["model.shared.weight"].numpy(), before["model.shared.weight"].numpy())
