"""CPU tests of CorrectBart beam search (DESIGN.md §3.12): the fp32 beam oracle against transformers'
generate(num_beams=K) token for token, the beam settings the library rejects, and the ctypes layout of
pllb_beam_desc."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from asr_rescoring_b200 import _lib, engine  # noqa: E402
from oracle import bart_beam_oracle as bb  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402

CLS, SEP = 101, 102
BASE = dict(max_length=12, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)


def _tiny(eos_bias=0.0, seed=3):
    import torch
    cfg = bo.bart_config(d_model=256, layers=2, ffn=512, vocab=300, max_position=64)
    m = bo.make_model(cfg, seed=seed)
    with torch.no_grad():
        m.final_logits_bias[0, SEP] += eos_bias
    return cfg, m


def _sents(n, seed=1):
    rng = np.random.default_rng(seed)
    return [[int(x) for x in rng.integers(104, 300, size=int(L))] for L in rng.integers(0, 14, size=n)]


def _check_against_generate(m, sents, gen):
    bs = bb.beam(m, sents, CLS, SEP, gen)
    ids, lens, sc = bs.result()
    ref, ref_sc = bb.hf_beam(m, sents, CLS, SEP, gen)
    K = gen["num_beams"]
    for i in range(len(sents)):
        for k in range(K):
            assert abs(float(sc[i, k]) - float(ref_sc[i, k])) <= 1e-5, (i, k, sc[i, k], ref_sc[i, k])
            assert (ids[i, k, lens[i, k]:] == 0).all()
            # slots left at the -1e9 start score (forced EOS at max_length 2) tie exactly with -1e9 candidates:
            # torch.topk leaves their order unspecified, the contract keeps the old slot
            if ref_sc[i, k] > bb.DEAD:
                assert ids[i, k, :lens[i, k]].tolist() == ref[i][k], (i, k)
    return lens


@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("lp", [1.0, 0.5, 2.0, 0.0])
@pytest.mark.parametrize("es", [False, True, "never"])
def test_beam_oracle_matches_generate(K, lp, es):
    # the EOS-favouring bias makes hypotheses finish at different steps
    cfg, m = _tiny(eos_bias=3.0)
    gen = dict(BASE, num_beams=K, num_return_sequences=K, length_penalty=lp, early_stopping=es)
    lens = _check_against_generate(m, _sents(6), gen)
    if lp <= 1.0:                     # a strong length penalty favours the longest hypotheses
        assert len(set(lens.ravel().tolist())) > 1


@pytest.mark.parametrize("case", ["no_bias", "forced", "max_length_2", "forced_max_length_2"])
def test_beam_oracle_edge_cases(case):
    cfg, m = _tiny(eos_bias=0.0 if case == "no_bias" else 3.0)
    gen = dict(BASE, num_beams=4, num_return_sequences=4, length_penalty=1.0, early_stopping=False)
    if case.startswith("forced"):
        gen.update(forced_bos_token_id=7, forced_eos_token_id=SEP)
    if case.endswith("max_length_2"):
        gen.update(max_length=2)
    sents = _sents(5, seed=2)
    lens = _check_against_generate(m, sents, gen)
    if case.endswith("max_length_2"):
        assert (lens[:, 0] == 2).all()
    if case == "forced":
        ids, lens, _ = bb.beam(m, sents, CLS, SEP, gen).result()
        assert (ids[:, :, 1] == 7).all()
        assert all(ids[i, k, lens[i, k] - 1] == SEP for i in range(5) for k in range(4))


def test_beam_select_margins_are_recorded():
    cfg, m = _tiny(eos_bias=3.0)
    gen = dict(BASE, num_beams=4, num_return_sequences=2, length_penalty=1.0, early_stopping=False)
    bs = bb.beam(m, _sents(3), CLS, SEP, gen)
    bs.result()
    kinds = {k for ms in bs.margins for _, k, _ in ms}
    assert {"2K cut", "running cut", "running order", "finished cut", "final order"} <= kinds
    assert len(bs.parents) == len(bs.run_scores) >= 1


@pytest.mark.parametrize("bad", [dict(num_beams=1), dict(num_beams=9), dict(num_return_sequences=0),
                                 dict(num_return_sequences=5), dict(length_penalty=float("inf")),
                                 dict(length_penalty=float("nan")), dict(early_stopping="always"),
                                 dict(do_sample=True), dict(no_repeat_ngram_size=3), dict(min_length=2),
                                 dict(repetition_penalty=1.2), dict(max_length=1), dict(max_length=65),
                                 dict(eos_token_id=300), dict(forced_bos_token_id=300)])
def test_beam_settings_rejections(bad):
    cfg, _ = _tiny()
    d = cfg.to_dict()
    good = dict(BASE, num_beams=4)
    g = engine.beam_settings(d, **good)
    assert g["num_return_sequences"] == 1 and g["length_penalty"] == 1.0 and g["early_stopping"] is False
    with pytest.raises(ValueError):
        engine.beam_settings(d, **dict(good, **bad))


def test_beam_settings_read_the_config():
    cfg, _ = _tiny()
    d = dict(cfg.to_dict(), num_beams=4, length_penalty=0.5, early_stopping="never")
    g = engine.beam_settings(d, **BASE)
    assert (g["num_beams"], g["length_penalty"], g["early_stopping"]) == (4, 0.5, "never")
    assert engine._beam_desc(g).early_stopping == 2
    assert engine._beam_desc(dict(g, early_stopping=True)).early_stopping == 1
    with pytest.raises(ValueError):
        engine.beam_settings(dict(d, vocab_size=7), **BASE)        # vocab < 2 * num_beams
    # greedy settings still refuse beams, also when the config carries them
    with pytest.raises(ValueError):
        engine.generation_settings(d, **BASE)
    with pytest.raises(ValueError):
        engine.generation_settings(cfg.to_dict(), **dict(BASE, num_beams=4))


def test_beam_desc_layout():
    assert ctypes.sizeof(_lib.BeamDesc) == 12
    assert [(n, getattr(_lib.BeamDesc, n).offset) for n, _ in _lib.BeamDesc._fields_] == [
        ("num_return_sequences", 0), ("length_penalty", 4), ("early_stopping", 8)]
