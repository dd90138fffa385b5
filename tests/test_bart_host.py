"""CPU tests of the CorrectBart path (DESIGN.md §3.11): the greedy oracle against generate(), the BART
state_dict mapping, the generation settings the library rejects, text decoding and the ctypes layout of
the seq2seq structs of include/pllb.h."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from asr_rescoring_b200 import _lib, engine  # noqa: E402
from asr_rescoring_b200.CorrectBart import model as cb  # noqa: E402
from asr_rescoring_b200.tokenizer import BertCharTokenizer  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402

CLS, SEP = 101, 102


def _tiny(seed=3, **kw):
    cfg = bo.bart_config(d_model=256, layers=2, ffn=512, vocab=300, max_position=64, **kw)
    return cfg, bo.make_model(cfg, seed=seed)


def _sents(n, vocab, seed=0, lens=None):
    rng = np.random.default_rng(seed)
    lens = lens if lens is not None else rng.integers(0, 14, size=n)
    return [[int(x) for x in rng.integers(104, vocab, size=int(L))] for L in lens]


@pytest.mark.parametrize("case", ["plain", "forced", "eos_bias", "scaled"])
def test_oracle_matches_generate(case):
    import torch
    cfg, m = _tiny(seed=3, scale_embedding=case == "scaled")
    gen = dict(max_length=12, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)
    if case == "forced":
        gen.update(forced_bos_token_id=7, forced_eos_token_id=SEP)
    if case == "eos_bias":
        with torch.no_grad():
            m.final_logits_bias[0, SEP] += 3.0      # sentences finish at different steps
    sents = _sents(8, 300, seed=1)
    ref = bo.hf_generate(m, sents, CLS, SEP, gen)
    ids, lens, _ = bo.greedy(m, sents, CLS, SEP, gen)
    for i in range(len(sents)):
        assert ids[i, :lens[i]].tolist() == ref[i]
        assert (ids[i, lens[i]:] == 0).all()                       # pad after EOS
    if case == "forced":
        assert (ids[:, 1] == 7).all() and all(r[-1] == SEP for r in ref)
    if case == "eos_bias":
        assert len(set(lens.tolist())) > 1                          # early EOS at different steps


def test_teacher_forced_logits_match_greedy_choices():
    cfg, m = _tiny(seed=4)
    gen = dict(max_length=10, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)
    sents = _sents(3, 300, seed=2)
    ids, lens, lg = bo.greedy(m, sents, CLS, SEP, gen)
    for i, s in enumerate(sents):
        tf = bo.teacher_forced_logits(m, s, ids[i, :lens[i]], CLS, SEP)
        for t in range(1, lens[i]):
            assert int(np.argmax(tf[t - 1])) == ids[i, t]
            assert abs(tf[t - 1, ids[i, t]] - lg[i, t]) < 1e-4


def test_state_dict_mapping_prefix_and_tied_keys():
    import torch
    cfg, m = _tiny()
    d = cfg.to_dict()
    sd = m.state_dict()
    keys = engine.bart_weight_keys(d)
    assert set(keys.values()) <= set(sd)
    used = set(keys.values()) | set(engine.BART_TIED_KEYS)
    assert set(sd) <= used, sorted(set(sd) - used)
    wrapped = {"bart." + k: v for k, v in sd.items()}
    got = engine.bart_state_dict(wrapped)
    assert set(got) == set(sd) and torch.equal(got["model.shared.weight"], sd["model.shared.weight"])
    untied = dict(sd)
    untied["lm_head.weight"] = sd["model.shared.weight"] + 1
    with pytest.raises(ValueError):
        engine.bart_state_dict(untied)
    with pytest.raises(ValueError):
        engine.bart_state_dict({k: v for k, v in sd.items() if k != "model.shared.weight"})
    shape = engine.check_bart_config(d)
    assert shape["hidden"] == 256 and shape["num_heads"] == 4 and shape["embed_scale"] == 1.0
    assert engine.check_bart_config(dict(d, scale_embedding=True))["embed_scale"] == 16.0
    with pytest.raises(ValueError):
        engine.check_bart_config(dict(d, activation_function="relu"))
    with pytest.raises(ValueError):
        engine.check_bart_config(dict(d, d_model=320, encoder_attention_heads=5, decoder_attention_heads=5))


@pytest.mark.parametrize("bad", [dict(num_beams=4), dict(do_sample=True), dict(no_repeat_ngram_size=3),
                                 dict(repetition_penalty=1.2), dict(min_length=5), dict(max_length=1),
                                 dict(max_length=65), dict(eos_token_id=300), dict(pad_token_id=-1),
                                 dict(decoder_start_token_id=1000), dict(forced_bos_token_id=300),
                                 dict(forced_eos_token_id=-5)])
def test_generation_settings_rejections(bad):
    cfg, _ = _tiny()
    d = cfg.to_dict()
    base = dict(max_length=20, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)
    engine.generation_settings(d, **base)
    with pytest.raises(ValueError):
        engine.generation_settings(d, **dict(base, **bad))


def test_decode_joins_without_spaces(tmp_path):
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]", "今", "天", "##ab", "ok"]
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tok = BertCharTokenizer(str(p))
    assert tok.decode([2, 104, 105, 106, 107, 102, 0, 0], skip_ids=[0, 2, 101, 102]) == "今天abok"
    assert tok.decode([101, 104, 102]) == "今"
    assert tok.decode([]) == ""


def test_compute_cer_and_one_hyp_shape():
    assert cb.one_hyp({"u1": {"hyp_1": "甲乙", "hyp_2": "x"}, "u2": {"hyp_1": "丙"}}) == ["甲乙", "丙"]
    with pytest.raises(ValueError):
        cb.compute_cer(["a"], [])


def _offsets(struct):
    return [(n, getattr(struct, n).offset) for n, _ in struct._fields_]


def test_s2s_struct_layout():
    """Sizes and field offsets of the seq2seq structs of include/pllb.h, written out by hand."""
    assert ctypes.sizeof(_lib.S2sDesc) == 56
    assert _offsets(_lib.S2sDesc) == [("enc_layers", 0), ("dec_layers", 4), ("hidden", 8), ("num_heads", 12),
                                      ("enc_intermediate", 16), ("dec_intermediate", 20), ("vocab", 24),
                                      ("enc_max_position", 28), ("dec_max_position", 32), ("ln_eps", 36),
                                      ("embed_scale", 40), ("cls_id", 44), ("sep_id", 48), ("operand_dtype", 52)]
    assert ctypes.sizeof(_lib.DecLayerWeights) == 26 * 8
    assert _offsets(_lib.DecLayerWeights) == [(n, 8 * i) for i, n in enumerate(
        ["q_w", "q_b", "k_w", "k_b", "v_w", "v_b", "o_w", "o_b", "self_ln_g", "self_ln_b",
         "cq_w", "cq_b", "ck_w", "ck_b", "cv_w", "cv_b", "co_w", "co_b", "cross_ln_g", "cross_ln_b",
         "ff1_w", "ff1_b", "ff2_w", "ff2_b", "final_ln_g", "final_ln_b"])]
    assert ctypes.sizeof(_lib.S2sWeights) == 144
    assert _offsets(_lib.S2sWeights) == [("enc", 0), ("dec_layers", 96), ("shared", 104), ("dec_pos_emb", 112),
                                         ("dec_emb_ln_g", 120), ("dec_emb_ln_b", 128), ("final_logits_bias", 136)]
    assert ctypes.sizeof(_lib.GenDesc) == 44
    assert _offsets(_lib.GenDesc) == [("max_length", 0), ("decoder_start_id", 4), ("eos_id", 8), ("pad_id", 12),
                                      ("forced_bos_id", 16), ("forced_eos_id", 20), ("num_beams", 24),
                                      ("do_sample", 28), ("no_repeat_ngram_size", 32), ("min_length", 36),
                                      ("repetition_penalty", 40)]
    assert ctypes.sizeof(_lib.S2sStats) == 64
    assert _offsets(_lib.S2sStats) == [("kernel_launches", 0), ("steps", 8), ("chunks", 16), ("sentences", 24),
                                       ("gemm_flops", 32), ("enc_ms", 40), ("cross_kv_ms", 44),
                                       ("dec_layers_ms", 48), ("head_ms", 52), ("total_ms", 56)]
