"""Beam search on the device (pllb_generate_beam, DESIGN.md §3.12) against the fp32 beam oracle
(oracle/bart_beam_oracle.py, pinned to transformers' generate(num_beams=K) by tests/test_bart_beam_host.py).

* Replay: the LM head and the selection alone (pllb_s2s_debug_beam_replay) on seeded hidden states,
  with logits recomputed on the host from the same 16-bit operands: every step of a sentence before its
  first decision with an oracle margin <= 1e-3 must match (parents, running scores within 1e-5), and a
  sentence without one must match in every hypothesis, scores within 1e-5.
* Teacher-forced: the oracle rescores every returned hypothesis; the device score must agree within a
  per-token tolerance per shape and operand type (random-init logit errors make identity no general gate).
* Identity: sentences whose output-deciding oracle margins all exceed 2 t eps (eps the per-token score
  tolerance; normalised for length-penalised comparisons) must equal generate() in all r hypotheses."""
import ctypes
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

from asr_rescoring_b200 import _lib, engine, synth  # noqa: E402
from oracle import bart_beam_oracle as bb  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402

CLS, SEP = 101, 102
# per-token tolerance of the teacher-forced score sum: measured worst case with headroom (DESIGN.md §3.12;
# measured 0.047 / 0.0055 / 0.51 / 0.052 on one B200)
SCORE_TOL = {("tiny", "bf16"): 0.08, ("tiny", "fp16"): 0.012, ("base", "bf16"): 0.8, ("base", "fp16"): 0.1}
# margins that only order running beams or finished slots among themselves decide no output
ORDER_ONLY = ("running order", "finished order")
GEN = dict(max_length=24, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0)


def _cache():
    if not hasattr(_cache, "d"):
        _cache.d = {}
    return _cache.d


def tiny(eos_bias=0.0):
    key = ("tiny", eos_bias)
    if key not in _cache():
        import torch
        cfg = bo.bart_config(d_model=256, layers=2, ffn=512, vocab=300, max_position=64)
        m = bo.make_model(cfg, seed=3)
        with torch.no_grad():
            m.final_logits_bias[0, SEP] += eos_bias
        _cache()[key] = (cfg, m)
    return _cache()[key]


def base():
    key = ("base",)
    if key not in _cache():
        cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512)
        _cache()[key] = (cfg, bo.make_model(cfg, seed=5))
    return _cache()[key]


def generator(shape, dtype, eos_bias=0.0, max_rows=0):
    key = ("gen", shape, dtype, eos_bias, max_rows)
    if key not in _cache():
        cfg, m = tiny(eos_bias) if shape == "tiny" else base()
        _cache()[key] = engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0, operand_dtype=dtype,
                                                max_rows=max_rows)
    return _cache()[key]


def pack(sents):
    off = np.zeros(len(sents) + 1, np.int64)
    np.cumsum([len(s) for s in sents], out=off[1:])
    tok = np.array([t for s in sents for t in s], np.int32)
    return tok, off


def rand_sents(n, vocab, seed, lo=0, hi=14):
    rng = np.random.default_rng(seed)
    return [[int(x) for x in rng.integers(104, vocab, size=int(L))] for L in rng.integers(lo, hi + 1, size=n)]


def c2_sents(n):
    nb = synth.make_nbest(n, 10)
    return [[synth.synthetic_token_id(c) for c in hs[0]] for hs in nb.hyps]


def settings(cfg, **kw):
    return engine.beam_settings(cfg.to_dict(), **dict(GEN, **kw))


def round16(x, dtype):
    import torch
    t = torch.as_tensor(np.asarray(x, np.float32))
    return t.to(torch.bfloat16 if dtype == "bf16" else torch.float16).float().numpy()


# ------------------------------------------------------------------------------------------ replay
def replay_case(shape, dtype, K, lp, es, forced=False, ml=12, n=16, seed=0):
    cfg, m = tiny() if shape == "tiny" else base()
    g = generator(shape, dtype)
    extra = dict(forced_bos_token_id=7, forced_eos_token_id=SEP) if forced else {}
    st = settings(cfg, num_beams=K, num_return_sequences=K, length_penalty=lp, early_stopping=es, max_length=ml,
                  **extra)
    H = cfg.d_model
    W = round16(m.model.shared.weight.detach().float().numpy(), dtype).astype(np.float64)
    bias = m.final_logits_bias.detach().float().numpy()[0].astype(np.float64)
    rng = np.random.default_rng(seed)
    hid = rng.standard_normal((ml - 1, n * K, H)).astype(np.float32) * 3.0
    # crafted steps that favour EOS: sentences finish at different steps
    eos_dir = W[SEP] / np.linalg.norm(W[SEP])
    for t in range(1, ml):
        rows = rng.random(n * K) < 0.25
        hid[t - 1, rows] += (rng.random((int(rows.sum()), 1)) * 12.0 * eos_dir).astype(np.float32)
    hid = round16(hid, dtype)
    ids, lens, sc, par, rs = g.debug_beam_replay(hid, st)
    bs = bb.BeamSearch(n, st)
    for t in range(1, ml):
        logits = (hid[t - 1].astype(np.float64) @ W.T + bias).astype(np.float32)
        bs.select(logits, t)
        if bs.done(t):
            break
    oi, ol, osc = bs.result()
    # every step before a sentence's first decision with margin <= 1e-3 must match; the outputs when there is none
    n_steps = n_full = 0
    for i in range(n):
        first = min([t for t, _, mg in bs.margins[i] if mg <= 1e-3], default=None)
        rows = slice(i * K, (i + 1) * K)
        for s, (p_o, r_o) in enumerate(zip(bs.parents, bs.run_scores)):
            if (first is not None and s + 1 >= first) or par[s, 0] < 0:
                break
            assert np.array_equal(par[s, rows], p_o[rows]), (i, s + 1)
            np.testing.assert_allclose(rs[s, rows], r_o[rows], rtol=1e-5, atol=1e-5)
            n_steps += 1
        if first is None:
            n_full += 1
            for k in range(K):
                assert lens[i, k] == ol[i, k], (i, k)
                assert ids[i, k, :lens[i, k]].tolist() == oi[i, k, :ol[i, k]].tolist(), (i, k)
                assert abs(float(sc[i, k]) - float(osc[i, k])) <= 1e-5 * max(1.0, abs(float(osc[i, k]))), (i, k)
    print(f"[replay {shape} {dtype} K={K} lp={lp} es={es} forced={forced} ml={ml}] {n_full} of {n} sentences "
          f"with every margin > 1e-3; {n_steps} sentence-steps checked; {len(bs.parents)} steps, "
          f"lengths {sorted(set(ol[:, 0].tolist()))}")
    assert n_steps > 0
    return n_full


@pytest.mark.parametrize("K", [2, 4, 8])
@pytest.mark.parametrize("lp", [1.0, 0.5, 2.0, 0.0])
@pytest.mark.parametrize("es", [False, True, "never"])
def test_replay_selection(K, lp, es):
    replay_case("tiny", "bf16", K, lp, es, seed=K * 7 + int(lp * 4))


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("case", ["forced", "max_length_2", "base_vocab"])
def test_replay_edge_cases(dtype, case):
    if case == "forced":
        replay_case("tiny", dtype, 4, 1.0, False, forced=True)
    elif case == "max_length_2":
        replay_case("tiny", dtype, 4, 1.0, False, forced=False, ml=2)
        replay_case("tiny", dtype, 8, 1.0, True, forced=True, ml=2)
    else:
        replay_case("base", dtype, 4, 1.0, False, ml=10, n=6)
        replay_case("base", dtype, 8, 0.5, "never", ml=10, n=6)


# ------------------------------------------------------------------------- end to end vs the oracle
def teacher_forced(m, sents, ids, lens, scores, st, tol, label):
    """Worst per-token |device score sum - oracle rescoring| over the returned hypotheses."""
    lp, ML = st["length_penalty"], st["max_length"]
    fb, fe = st.get("forced_bos_token_id"), st.get("forced_eos_token_id")
    worst = 0.0
    for i, s in enumerate(sents):
        for k in range(ids.shape[1]):
            L = int(lens[i, k])
            if scores[i, k] <= bb.DEAD or L < 2:
                continue
            seq = ids[i, k, :L]
            tf = bo.teacher_forced_logits(m, s, seq, CLS, SEP).astype(np.float64)
            lse = np.log(np.exp(tf - tf.max(1, keepdims=True)).sum(1)) + tf.max(1)
            tot = 0.0
            for t in range(1, L):
                forced = (t == ML - 1 and fe is not None) or (t == 1 and fb is not None)
                tot += 0.0 if forced else tf[t - 1, seq[t]] - lse[t - 1]
            dev = float(scores[i, k]) * float(L - 1) ** lp
            worst = max(worst, abs(dev - tot) / (L - 1))
    print(f"[{label}] worst per-token |device - oracle| score = {worst:.4g} (tolerance {tol})")
    assert worst <= tol, f"{label}: {worst} > {tol}"
    return worst


def identity(m, sents, ids, lens, st, eps, label):
    """Sentences whose output-deciding oracle margins all exceed what a per-token score error eps can
    flip equal generate() in every hypothesis: 2 t eps for cumulative scores at step t, 2 t eps / t^lp for
    length-normalised ones, 2 eps max(1, (ML - 1)^(1 - lp)) for the final order."""
    lp, ML = float(st["length_penalty"]), int(st["max_length"])

    def need(t, kind):
        if kind in ("2K cut", "K cut of the 2K", "running cut"):
            return 2 * t * eps
        if kind == "final order":
            return 2 * eps * max(1.0, float(ML - 1) ** (1 - lp))
        return 2 * t * eps / float(t) ** lp

    bs = bb.beam(m, sents, CLS, SEP, st)
    bs.result()
    ref, _ = bb.hf_beam(m, sents, CLS, SEP, dict(st, num_return_sequences=st["num_beams"]))
    n_sure = 0
    for i in range(len(sents)):
        if any(mg <= need(t, k) for t, k, mg in bs.margins[i] if k not in ORDER_ONLY):
            continue
        n_sure += 1
        for k in range(ids.shape[1]):
            assert ids[i, k, :lens[i, k]].tolist() == ref[i][k], f"{label}: sentence {i} hypothesis {k}"
    print(f"[{label}] identity with generate(): {n_sure} of {len(sents)} sentences certified (eps = {eps})")
    return n_sure


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_tiny_teacher_forced_and_identity(dtype):
    cfg, m = tiny(eos_bias=1.5)
    sents = rand_sents(80, 300, seed=11)
    for K, r, lp, es in ((4, 4, 1.0, False), (2, 1, 0.5, True), (8, 3, 2.0, "never")):
        st = settings(cfg, num_beams=K, num_return_sequences=r, length_penalty=lp, early_stopping=es)
        ids, lens, sc = generator("tiny", dtype, eos_bias=1.5).beam_search_packed(*pack(sents), st)
        label = f"tiny {dtype} K={K} r={r} lp={lp} es={es}"
        teacher_forced(m, sents, ids, lens, sc, st, SCORE_TOL[("tiny", dtype)], label)
        n_sure = identity(m, sents, ids, lens, st, SCORE_TOL[("tiny", dtype)], label)
        if dtype == "fp16" and K == 4:
            assert n_sure > 0


@pytest.mark.parametrize("dtype", ["bf16", "fp16"])
def test_base_shape_c2_sentences(dtype):
    cfg, m = base()
    sents = c2_sents(60)
    st = settings(cfg, num_beams=4, num_return_sequences=4, max_length=50)
    ids, lens, sc = generator("base", dtype).beam_search_packed(*pack(sents), st)
    label = f"base {dtype} K=4"
    teacher_forced(m, sents[:24], ids[:24], lens[:24], sc[:24], st, SCORE_TOL[("base", dtype)], label)
    identity(m, sents[:12], ids[:12], lens[:12], st, SCORE_TOL[("base", dtype)], label + " (first 12)")


def test_forced_and_early_eos():
    import torch  # noqa: F401
    cfg, m = tiny(eos_bias=3.0)
    sents = rand_sents(16, 300, seed=5) + [[]]
    st = settings(cfg, num_beams=4, num_return_sequences=2, max_length=10, forced_bos_token_id=7,
                  forced_eos_token_id=SEP)
    ids, lens, sc = generator("tiny", "fp16", eos_bias=3.0).beam_search_packed(*pack(sents), st)
    assert (ids[:, :, 1] == 7).all()
    for i in range(len(sents)):
        for k in range(2):
            assert ids[i, k, lens[i, k] - 1] == SEP and (ids[i, k, lens[i, k]:] == 0).all()
    assert (np.diff(sc, axis=1) <= 0).all()
    teacher_forced(m, sents, ids, lens, sc, st, SCORE_TOL[("tiny", "fp16")], "forced fp16")
    st2 = settings(cfg, num_beams=4, num_return_sequences=4, max_length=2)
    ids, lens, sc = generator("tiny", "fp16", eos_bias=3.0).beam_search_packed(*pack(sents), st2)
    assert ids.shape == (len(sents), 4, 2) and (lens[:, 0] == 2).all() and (ids[:, :, 0] == 2).all()


def test_bitwise_invariance_runs_and_max_rows():
    cfg, m = tiny(eos_bias=1.5)
    sents = rand_sents(37, 300, seed=7)
    K = 4
    st = settings(cfg, num_beams=K, num_return_sequences=K, length_penalty=0.5)
    ref = generator("tiny", "bf16", eos_bias=1.5).beam_search_packed(*pack(sents), st)
    again = generator("tiny", "bf16", eos_bias=1.5).beam_search_packed(*pack(sents), st)
    for a, b in zip(ref, again):
        assert np.array_equal(a, b)
    # max_rows = K decodes every sentence alone: a frozen sentence's result does not depend on its companions
    for max_rows in (0, K, 5 * K, 16 * K):
        with engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0, max_rows=max_rows) as g:
            got = g.beam_search_packed(*pack(sents), st)
        for a, b in zip(ref, got):
            assert np.array_equal(a, b), f"max_rows={max_rows}"


def test_library_rejects_unsupported_beam_settings():
    cfg, m = tiny()
    g = generator("tiny", "bf16")
    good = settings(cfg, num_beams=4, num_return_sequences=2)
    tok, off = pack([[104, 105]])

    def rc_of(gen, beam, handle=None):
        ids = np.zeros(8 * 64, np.int32)
        ln = np.zeros(8, np.int32)
        sc = np.zeros(8, np.float32)
        return g._lib.pllb_generate_beam_host(handle or g._h, ctypes.byref(gen), ctypes.byref(beam), engine._np_ptr(tok),
                                              engine._np_ptr(off), 1, engine._np_ptr(ids), engine._np_ptr(ln),
                                              engine._np_ptr(sc))

    assert rc_of(engine._gen_desc(good), engine._beam_desc(good)) == 0
    for bad in (dict(num_beams=1), dict(num_beams=9), dict(do_sample=True), dict(no_repeat_ngram_size=2),
                dict(min_length=3), dict(repetition_penalty=1.5), dict(max_length=1), dict(max_length=65),
                dict(eos_token_id=300), dict(forced_bos_token_id=300)):
        assert rc_of(engine._gen_desc(dict(good, **bad)), engine._beam_desc(good)) == 1, bad
    for bad in (dict(num_return_sequences=0), dict(num_return_sequences=5), dict(length_penalty=float("inf"))):
        assert rc_of(engine._gen_desc(good), engine._beam_desc(dict(good, **bad))) == 1, bad
    b = engine._beam_desc(good)
    b.early_stopping = 3
    assert rc_of(engine._gen_desc(good), b) == 1
    # greedy still refuses beams, and a chunk must hold one sentence's beams
    d = engine._gen_desc(good)
    rc = g._lib.pllb_generate_host(g._h, ctypes.byref(d), engine._np_ptr(tok), engine._np_ptr(off), 1,
                                   engine._np_ptr(np.zeros(64, np.int32)), engine._np_ptr(np.zeros(1, np.int32)), None)
    assert rc == 1
    with engine.Seq2SeqGenerator(m.state_dict(), cfg.to_dict(), device=0, max_rows=3) as small:
        assert rc_of(engine._gen_desc(good), engine._beam_desc(good), small._h) == 1
    with pytest.raises(_lib.PllbError):
        g.beam_search_packed(np.array([300], np.int32), np.array([0, 1], np.int64), good)


def test_correct_bart_beam_end_to_end(tmp_path):
    from asr_rescoring_b200.CorrectBart.model import CorrectBart, compute_cer
    from asr_rescoring_b200.tokenizer import BertCharTokenizer
    cfg, m = tiny(eos_bias=1.5)
    chars = [chr(0x4E00 + 37 * i) for i in range(196)]
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"] + chars
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tok = BertCharTokenizer(str(p))
    rng = np.random.default_rng(8)
    texts = ["".join(rng.choice(chars, size=int(L))) for L in rng.integers(1, 12, size=24)]
    refs = ["".join(rng.choice(chars, size=int(L))) for L in rng.integers(1, 12, size=24)]
    model = CorrectBart(m.state_dict(), cfg.to_dict(), tok, device=0, max_length=20, operand_dtype="fp16",
                        generation=dict(decoder_start_token_id=2, num_beams=4))
    try:
        assert model.beam and model.generation["num_beams"] == 4
        preds = model.correct(texts)
        sents = [tok.encode(t) for t in texts]
        ids, lens = model.generate_packed(*pack(sents))
    finally:
        model.close()
    bs = bb.beam(m, sents, CLS, SEP, model.generation)
    oi, ol, _ = bs.result()
    same = [i for i in range(len(texts)) if ids[i, :lens[i]].tolist() == oi[i, 0, :ol[i, 0]].tolist()]
    print(f"[correct beam] {len(same)} of {len(texts)} best hypotheses token-identical to the oracle")
    assert len(same) > 0
    skip = model.skip_ids()
    for i in same:
        assert preds[i] == tok.decode(oi[i, 0, :ol[i, 0]], skip)
    got = compute_cer([preds[i] for i in same], [refs[i] for i in same])
    exp = sum(_lev(refs[i], preds[i]) for i in same) / sum(len(refs[i]) for i in same)
    assert got == pytest.approx(exp, abs=1e-12)


def _lev(a, b):
    d = list(range(len(b) + 1))
    for i in range(1, len(a) + 1):
        prev, d[0] = d[0], i
        for j in range(1, len(b) + 1):
            cur = min(d[j] + 1, d[j - 1] + 1, prev + (a[i - 1] != b[j - 1]))
            prev, d[j] = d[j], cur
    return d[len(b)]
