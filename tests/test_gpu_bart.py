"""Greedy BART generation on the device (pllb_generate, DESIGN.md §3.11) against the fp32 CPU oracle
(oracle/bart_oracle.py, itself pinned to transformers' generate() by tests/test_bart_host.py).

Acceptance is teacher-forced: the oracle runs on the device's OWN output sequence and every emitted
token d must satisfy |device logit - l_oracle[d]| <= delta and l_oracle[d] >= max l_oracle - 2 delta
(random-init logits have small top-2 gaps, so identity cannot be the general gate).  Sentences whose
oracle path has a top-2 margin > 4 delta at every step must match generate() exactly."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

from asr_rescoring_b200 import _lib, engine, synth  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402

CLS, SEP = 101, 102
# logit tolerance per (shape, operand type): measured worst case with headroom (DESIGN.md §3.11)
DELTA = {("tiny", "bf16"): 0.25, ("tiny", "fp16"): 0.06, ("base", "bf16"): 1.0, ("base", "fp16"): 0.25}
GEN = dict(max_length=24, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)


def _models():
    if not hasattr(_models, "cache"):
        _models.cache = {}
    return _models.cache


def tiny(scale=False, seed=3):
    key = ("tiny", scale, seed)
    if key not in _models():
        cfg = bo.bart_config(d_model=256, layers=2, ffn=512, vocab=300, max_position=64, scale_embedding=scale)
        _models()[key] = (cfg, bo.make_model(cfg, seed=seed))
    return _models()[key]


def base():
    key = ("base",)
    if key not in _models():
        cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512)
        _models()[key] = (cfg, bo.make_model(cfg, seed=5))
    return _models()[key]


def pack(sents):
    off = np.zeros(len(sents) + 1, np.int64)
    np.cumsum([len(s) for s in sents], out=off[1:])
    tok = np.array([t for s in sents for t in s], np.int32)
    return tok, off


def device_generate(cfg, m, sents, gen, dtype, max_rows=0):
    with engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0, operand_dtype=dtype,
                                 max_rows=max_rows) as g:
        tok, off = pack(sents)
        return g.generate_packed(tok, off, engine.generation_settings(cfg.to_dict(), **gen), return_logits=True)


def rand_sents(n, vocab, seed, lo=0, hi=14):
    rng = np.random.default_rng(seed)
    return [[int(x) for x in rng.integers(104, vocab, size=int(L))] for L in rng.integers(lo, hi + 1, size=n)]


def c2_sents(n):
    nb = synth.make_nbest(n, 10)
    return [[synth.synthetic_token_id(c) for c in hs[0]] for hs in nb.hyps]


def accept(m, sents, ids, lens, lg, gen, delta, label):
    """Teacher-forced acceptance; returns (worst |dlogit|, worst gap below the max)."""
    worst_d = worst_gap = 0.0
    fb, fe, ML = gen.get("forced_bos_token_id"), gen.get("forced_eos_token_id"), gen["max_length"]
    for i, s in enumerate(sents):
        tf = bo.teacher_forced_logits(m, s, ids[i, :lens[i]], CLS, SEP)
        for t in range(1, lens[i]):
            d = ids[i, t]
            worst_d = max(worst_d, abs(float(lg[i, t]) - float(tf[t - 1, d])))
            forced = (t == ML - 1 and fe is not None) or (t == 1 and fb is not None)
            if not forced:
                worst_gap = max(worst_gap, float(tf[t - 1].max() - tf[t - 1, d]))
    print(f"[{label}] worst |device - oracle logit| = {worst_d:.4g}, worst gap below the max = {worst_gap:.4g}, "
          f"delta = {delta}")
    assert worst_d <= delta, f"{label}: logit error {worst_d} > {delta}"
    assert worst_gap <= 2 * delta, f"{label}: chosen token {worst_gap} below the max > {2 * delta}"
    return worst_d, worst_gap


def identity(m, sents, ids, lens, gen, delta, label):
    """Exact identity with generate() for sentences whose oracle path has top-2 margin > 4 delta."""
    oi, ol, _ = bo.greedy(m, sents, CLS, SEP, gen)
    ref = bo.hf_generate(m, sents, CLS, SEP, gen)
    n_sure = 0
    for i, s in enumerate(sents):
        assert oi[i, :ol[i]].tolist() == ref[i]
        tf = bo.teacher_forced_logits(m, s, oi[i, :ol[i]], CLS, SEP)
        top2 = np.sort(tf[:ol[i] - 1], axis=1)[:, -2:]
        if (top2[:, 1] - top2[:, 0] > 4 * delta).all():
            n_sure += 1
            assert ids[i, :lens[i]].tolist() == ref[i], f"{label}: sentence {i} differs from generate()"
    print(f"[{label}] exact identity with generate(): {n_sure} of {len(sents)} sentences have margin > 4 delta")
    return n_sure


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_tiny_teacher_forced_and_identity(dtype):
    cfg, m = tiny()
    sents = rand_sents(40, 300, seed=11)
    ids, lens, lg = device_generate(cfg, m, sents, GEN, dtype)
    delta = DELTA[("tiny", dtype)]
    accept(m, sents, ids, lens, lg, GEN, delta, f"tiny {dtype}")
    assert identity(m, sents, ids, lens, GEN, delta, f"tiny {dtype}") > 0


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_base_shape_c2_sentences(dtype):
    cfg, m = base()
    sents = c2_sents(200)
    gen = dict(GEN, max_length=50)
    ids, lens, lg = device_generate(cfg, m, sents, gen, dtype)
    delta = DELTA[("base", dtype)]
    accept(m, sents, ids, lens, lg, gen, delta, f"base {dtype}")
    identity(m, sents[:40], ids[:40], lens[:40], gen, delta, f"base {dtype} (first 40)")


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_edge_cases(dtype):
    import torch
    cfg, m = tiny()
    delta = DELTA[("tiny", dtype)]
    # empty input (T = 2) and an input at max_position
    sents = [[], rand_sents(1, 300, seed=2, lo=62, hi=62)[0], [105, 106]]
    ids, lens, lg = device_generate(cfg, m, sents, GEN, dtype)
    accept(m, sents, ids, lens, lg, GEN, delta, f"edge lengths {dtype}")
    with pytest.raises(_lib.PllbError) as e:
        device_generate(cfg, m, [[104] * 63], GEN, dtype)
    assert e.value.code == 5
    # max_length = 2
    g2 = dict(GEN, max_length=2)
    ids, lens, lg = device_generate(cfg, m, sents, g2, dtype)
    assert ids.shape == (3, 2) and (lens == 2).all() and (ids[:, 0] == 2).all()
    accept(m, sents, ids, lens, lg, g2, delta, f"max_length 2 {dtype}")
    # forced BOS / EOS
    gf = dict(GEN, max_length=10, forced_bos_token_id=7, forced_eos_token_id=SEP)
    s8 = rand_sents(8, 300, seed=4)
    ids, lens, lg = device_generate(cfg, m, s8, gf, dtype)
    assert (ids[:, 1] == 7).all() and all(ids[i, lens[i] - 1] == SEP for i in range(8))
    accept(m, s8, ids, lens, lg, gf, delta, f"forced {dtype}")
    # EOS-favouring bias: sentences finish at different steps; then all at step 1
    cfg_b = bo.bart_config(d_model=256, layers=2, ffn=512, vocab=300, max_position=64)
    mb = bo.make_model(cfg_b, seed=3)
    with torch.no_grad():
        mb.final_logits_bias[0, SEP] += 3.0
    s16 = rand_sents(16, 300, seed=5)
    ids, lens, lg = device_generate(cfg_b, mb, s16, GEN, dtype)
    accept(mb, s16, ids, lens, lg, GEN, delta, f"eos bias {dtype}")
    assert len(set(lens.tolist())) > 1
    for i in range(16):
        assert (ids[i, lens[i]:] == 0).all()
    with torch.no_grad():
        mb.final_logits_bias[0, SEP] += 100.0
    ids, lens, lg = device_generate(cfg_b, mb, s16, GEN, dtype)
    assert (lens == 2).all() and (ids[:, 1] == SEP).all() and (ids[:, 2:] == 0).all()


@pytest.mark.parametrize("scale", [False, True])
def test_scale_embedding(scale):
    cfg, m = tiny(scale=scale)
    sents = rand_sents(16, 300, seed=6)
    ids, lens, lg = device_generate(cfg, m, sents, GEN, "fp16")
    accept(m, sents, ids, lens, lg, GEN, DELTA[("tiny", "fp16")], f"scale_embedding={scale}")


def test_bitwise_invariance_runs_and_max_rows():
    cfg, m = tiny()
    sents = rand_sents(37, 300, seed=7)
    ref = device_generate(cfg, m, sents, GEN, "bf16")
    for max_rows in (0, 1, 5, 16):
        got = device_generate(cfg, m, sents, GEN, "bf16", max_rows=max_rows)
        for a, b in zip(ref, got):
            assert np.array_equal(a, b), f"max_rows={max_rows}"


def test_library_rejects_unsupported_generation():
    import ctypes
    cfg, m = tiny()
    with engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0) as g:
        good = engine.generation_settings(cfg.to_dict(), **GEN)
        tok, off = pack([[104, 105]])
        for bad in (dict(num_beams=2), dict(do_sample=True), dict(no_repeat_ngram_size=2), dict(min_length=3),
                    dict(repetition_penalty=1.5), dict(max_length=1), dict(max_length=65), dict(eos_token_id=300),
                    dict(forced_bos_token_id=300)):
            d = engine._gen_desc(dict(good, **bad))
            ids = np.zeros(64, np.int32)
            ln = np.zeros(1, np.int32)
            rc = g._lib.pllb_generate_host(g._h, ctypes.byref(d), engine._np_ptr(tok), engine._np_ptr(off), 1,
                                           engine._np_ptr(ids), engine._np_ptr(ln), None)
            assert rc == 1, bad
        with pytest.raises(_lib.PllbError):
            g.generate_packed(np.array([300], np.int32), np.array([0, 1], np.int64), good)


def test_correct_bart_end_to_end(tmp_path):
    from asr_rescoring_b200.CorrectBart.model import CorrectBart, compute_cer
    from asr_rescoring_b200.tokenizer import BertCharTokenizer
    cfg, m = tiny()
    chars = [chr(0x4E00 + 37 * i) for i in range(196)]
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"] + chars
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tok = BertCharTokenizer(str(p))
    rng = np.random.default_rng(8)
    texts = ["".join(rng.choice(chars, size=int(L))) for L in rng.integers(1, 12, size=24)]
    refs = ["".join(rng.choice(chars, size=int(L))) for L in rng.integers(1, 12, size=24)]
    model = CorrectBart(m.state_dict(), cfg.to_dict(), tok, device=0, max_length=20, operand_dtype="fp16",
                        generation=dict(decoder_start_token_id=2))
    try:
        preds = model.correct(texts)
        sents = [tok.encode(t) for t in texts]
        ids, lens = model.generate_packed(*pack(sents))
    finally:
        model.close()
    oi, ol, _ = bo.greedy(m, sents, CLS, SEP, model.generation)
    same = [i for i in range(len(texts)) if ids[i, :lens[i]].tolist() == oi[i, :ol[i]].tolist()]
    print(f"[correct] {len(same)} of {len(texts)} sentences token-identical to the oracle")
    assert len(same) > 0
    skip = model.skip_ids()
    o_text = [tok.decode(oi[i, :ol[i]], skip) for i in range(len(texts))]
    for i in same:
        assert preds[i] == o_text[i]
    got = compute_cer([preds[i] for i in same], [refs[i] for i in same])
    exp = sum(_lev(refs[i], o_text[i]) for i in same) / sum(len(refs[i]) for i in same)
    assert got == pytest.approx(exp, abs=1e-12)


def _lev(a, b):
    d = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        prev, d[0] = d[0], i
        for j in range(1, len(b) + 1):
            cur = min(d[j] + 1, d[j - 1] + 1, prev + (a[i - 1] != b[j - 1]))
            prev, d[j] = d[j], cur
    return d[len(b)]
