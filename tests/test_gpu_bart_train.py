"""CorrectBart fine-tuning on the device (pllb_s2s_train_*, DESIGN.md §3.13) against the fp32 CPU autograd
oracle (oracle/bart_train_oracle.py: transformers' forward(labels=...), backward and torch.optim.AdamW).

Parity is at dropout 0 with mode 2 (gradients without the update): the loss, the per-position losses and the
relative L2 error of every parameter's gradient.  The tolerances are the measured worst case with headroom
(DESIGN.md §3.13)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu

from asr_rescoring_b200 import _lib, engine, synth  # noqa: E402
from oracle import bart_oracle as bo  # noqa: E402
from oracle import bart_train_oracle as bto  # noqa: E402

CLS, SEP = 101, 102
# Measured worst case on a B200 with headroom (DESIGN.md §3.13, profiles/correct_bart_train_gpu_tests.log).
# Measured worst: loss 1.0e-3 / 5e-6, token 0.062 / 0.0087, gradient 0.055 / 0.0084, shared 0.032 / 0.0032.
LOSS_REL = {"tiny": 5e-3, "base": 1e-3}        # |loss - oracle| / oracle
TOKEN_ABS = {"tiny": 0.1, "base": 0.03}        # per-position loss, nats
GRAD_REL = {"tiny": 0.09, "base": 0.015}       # per-tensor relative L2 error of the gradient
# shared, whole and on the rows the decoder input looks up.  Leaving out the decoder lookup's contribution moves
# the tiny-shape figures to >= 0.087 and >= 0.137 (fp32 autograd with that contribution detached), so these
# bounds see each of shared's three contributions.
SHARED_REL = {"tiny": 0.05, "base": 0.01}


def tiny_model(scale=False, seed=3):
    cfg = bo.bart_config(d_model=256, layers=2, ffn=1024, vocab=300, max_position=64, scale_embedding=scale)
    return cfg, bo.make_model(cfg, seed=seed)


def batch(rng, B, Te, Td, V, label_pad=-100, pad_id=0):
    """Ragged encoder rows ([CLS] t [SEP]) and ragged labels ([CLS] t [SEP], then label_pad)."""
    ids = np.full((B, Te), pad_id, np.int64)
    mask = np.zeros((B, Te), np.int64)
    labels = np.full((B, Td), label_pad, np.int64)
    for b in range(B):
        ne = int(rng.integers(3, Te + 1)) if b else Te
        ids[b, :ne] = [CLS] + list(rng.integers(110, V, ne - 2)) + [SEP]
        mask[b, :ne] = 1
        nd = int(rng.integers(3, Td + 1)) if b else Td
        labels[b, :nd] = [CLS] + list(rng.integers(110, V, nd - 2)) + [SEP]
    return ids, mask, labels


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


def trainer(cfg, m, **kw):
    kw.setdefault("dropout", 0.0)
    kw.setdefault("attention_dropout", 0.0)
    kw.setdefault("max_batch", 8)
    kw.setdefault("max_enc_len", 32)
    kw.setdefault("max_dec_len", 32)
    return engine.Seq2SeqTrainer(m.state_dict(), cfg.to_dict(), device=0, **kw)


def check_parity(kind, cfg, m, ids, mask, labels):
    import copy
    ref = copy.deepcopy(m)
    loss_o, tl_o, g_o, _ = bto.step(ref, ids, mask, labels, update=False)
    with trainer(cfg, m, max_batch=ids.shape[0], max_enc_len=ids.shape[1], max_dec_len=labels.shape[1]) as tr:
        loss = tr.step(ids, mask, labels, mode=2)
        tl = tr.token_losses()
        g = tr.grads()
    assert abs(loss - loss_o) <= LOSS_REL[kind] * abs(loss_o), (loss, loss_o)
    assert np.all(tl[labels == -100] == 0.0)
    tok_err = float(np.abs(tl - tl_o).max())
    # k_proj.bias is left out: softmax is invariant to a key bias, so its exact gradient is 0 and both sides
    # hold rounding noise only
    errs = {k: rel_l2(g[k].numpy(), v.numpy()) for k, v in g_o.items()
            if float(v.abs().max()) > 0 and not k.endswith("k_proj.bias")}
    worst = max(errs, key=errs.get)
    print(f"[parity {kind}] loss {loss:.6f} vs {loss_o:.6f}; token |d| max {tok_err:.4f}; "
          f"grad rel L2 worst {errs[worst]:.4f} ({worst}), median {np.median(list(errs.values())):.4f}, "
          f"shared {errs['model.shared.weight']:.4f}")
    for k in sorted(errs, key=errs.get, reverse=True)[:12]:
        print(f"    {errs[k]:.4f}  {k}")
    rows = np.unique(engine.shift_tokens_right(labels, 0, cfg.decoder_start_token_id))
    rows = rows[rows != 0]                                   # the pad row gets nothing from the lookups
    dec_rows = rel_l2(g["model.shared.weight"].numpy()[rows], g_o["model.shared.weight"].numpy()[rows])
    print(f"    shared on the {len(rows)} decoder-input rows: {dec_rows:.4f}")
    assert tok_err <= TOKEN_ABS[kind]
    assert errs[worst] <= GRAD_REL[kind], (worst, errs[worst])
    assert errs["model.shared.weight"] <= SHARED_REL[kind] and dec_rows <= SHARED_REL[kind]
    for k in ("model.encoder.embed_positions.weight", "model.decoder.embed_positions.weight"):
        assert float(g[k][:2].abs().max()) == 0.0          # rows 0 and 1 are never looked up
    return errs


@pytest.mark.parametrize("scale", [False, True])
@pytest.mark.parametrize("label_pad", [-100, 0])
def test_parity_tiny(scale, label_pad):
    cfg, m = tiny_model(scale=scale)
    rng = np.random.default_rng(11 + scale + 2 * (label_pad == 0))
    ids, mask, labels = batch(rng, 5, 13, 9, 300, label_pad=label_pad)
    check_parity("tiny", cfg, m, ids, mask, labels)


def c2_pairs(n):
    from asr_rescoring_b200.tokenizer import SyntheticCharTokenizer
    nb = synth.make_nbest(n, 10, seed=0)
    return SyntheticCharTokenizer(), [hs[0] for hs in nb.hyps], list(nb.refs)


def test_parity_base_and_three_steps():
    import copy
    import torch
    from asr_rescoring_b200.CorrectBart.train import make_batches
    # transformers' default init_std 0.02: with the 0.1 of the tiny model the bf16 logits at this vocabulary are off
    # by up to 0.8 (DESIGN.md §3.11), which no softmax gradient survives
    cfg = bo.bart_config(d_model=768, layers=6, ffn=3072, vocab=21128, max_position=512, init_std=0.02)
    m = bo.make_model(cfg, seed=5)
    tok, hyps, refs = c2_pairs(32)
    b = make_batches(tok, hyps, refs, 32)[0]
    check_parity("base", cfg, m, b["input_ids"], b["attention_mask"], b["labels"])
    ref = copy.deepcopy(m)
    opt = torch.optim.AdamW(ref.parameters(), lr=1e-4, weight_decay=0.01)
    with trainer(cfg, m, lr=1e-4, max_batch=32, max_enc_len=b["input_ids"].shape[1],
                 max_dec_len=b["labels"].shape[1]) as tr:
        for k in range(3):
            lo = bto.step(ref, b["input_ids"], b["attention_mask"], b["labels"], optimizer=opt)[0]
            ld = tr.step(b["input_ids"], b["attention_mask"], b["labels"], mode=1)
            print(f"[base AdamW step {k}] device {ld:.5f} oracle {lo:.5f}")
            assert abs(ld - lo) <= LOSS_REL["base"] * lo


def test_export_and_optimizer():
    cfg, m = tiny_model()
    sd_in = m.state_dict()
    rng = np.random.default_rng(5)
    ids, mask, labels = batch(rng, 4, 10, 8, 300)
    with trainer(cfg, m, lr=1e-3) as tr:
        tr.step(ids, mask, labels, mode=0)
        out = tr.state_dict()
        assert list(out) == list(sd_in)
        for k, v in sd_in.items():
            assert np.array_equal(out[k].numpy(), v.numpy()), k          # mode 0 changes nothing
        for _ in range(2):
            tr.step(ids, mask, labels, mode=1)
        out = tr.state_dict()
    assert np.array_equal(out["final_logits_bias"].numpy(), sd_in["final_logits_bias"].numpy())
    assert not np.array_equal(out["model.shared.weight"].numpy(), sd_in["model.shared.weight"].numpy())
    for k in engine.BART_TIED_KEYS:
        if k in out:
            assert np.array_equal(out[k].numpy(), out["model.shared.weight"].numpy())
    pos = out["model.encoder.embed_positions.weight"].numpy()[:2]          # no gradient: AdamW only decays them
    np.testing.assert_allclose(pos, sd_in["model.encoder.embed_positions.weight"].numpy()[:2] * (1 - 1e-3 * 0.01) ** 2,
                               rtol=1e-6)
    with engine.Seq2SeqGenerator(out, cfg.to_dict(), device=0) as g:
        gi, gl = g.generate_packed(np.array([120, 130, 140], np.int32), np.array([0, 3], np.int64),
                                   dict(max_length=8, decoder_start_token_id=2, eos_token_id=SEP, pad_token_id=0))
    assert gi.shape == (1, 8) and 1 <= gl[0] <= 8


def _run(cfg, m, ids, mask, labels, n=3, **kw):
    with trainer(cfg, m, lr=1e-3, **kw) as tr:
        losses = [tr.step(ids, mask, labels, mode=1) for _ in range(n)]
        return losses, tr.state_dict(), tr.graph_replays()


def test_determinism_and_graphs(monkeypatch):
    cfg, m = tiny_model()
    rng = np.random.default_rng(6)
    ids, mask, labels = batch(rng, 4, 12, 10, 300)
    l1, s1, r1 = _run(cfg, m, ids, mask, labels, n=4, dropout=0.1, attention_dropout=0.1)
    l2, s2, _ = _run(cfg, m, ids, mask, labels, n=4, dropout=0.1, attention_dropout=0.1)
    assert l1 == l2 and all(np.array_equal(s1[k].numpy(), s2[k].numpy()) for k in s1)
    assert r1 == 3                       # eager, then capture + replay, replay, replay
    monkeypatch.setenv("PLLB_TRAIN_GRAPH", "0")
    l3, s3, r3 = _run(cfg, m, ids, mask, labels, n=4, dropout=0.1, attention_dropout=0.1)
    assert r3 == 0 and l3 == l1 and all(np.array_equal(s1[k].numpy(), s3[k].numpy()) for k in s1)


def test_dropout():
    cfg, m = tiny_model()
    rng = np.random.default_rng(7)
    ids, mask, labels = batch(rng, 4, 12, 10, 300)

    def losses(seed, mode):
        with trainer(cfg, m, dropout=0.3, attention_dropout=0.3, seed=seed) as tr:
            return [tr.step(ids, mask, labels, mode=mode) for _ in range(2)]
    a, b, c = losses(1, 2), losses(1, 2), losses(2, 2)
    assert a == b and a != c and np.all(np.isfinite(a + c))
    e0, e1 = losses(1, 0), losses(2, 0)
    assert e0 == e1 and e0[0] == e0[1]                # mode 0 bypasses dropout
    with trainer(cfg, m) as tr:
        assert tr.step(ids, mask, labels, mode=0) == e0[0]


def test_rejections():
    cfg, m = tiny_model()
    rng = np.random.default_rng(9)
    ids, mask, labels = batch(rng, 2, 8, 6, 300)
    with trainer(cfg, m, max_batch=2, max_enc_len=8, max_dec_len=6) as tr:
        lib, h = tr._lib, tr._h

        def code(i=ids, nv=None, lab=labels, B=2, Te=8, Td=6, mode=2):
            i = np.ascontiguousarray(i, np.int32)
            lab = np.ascontiguousarray(lab, np.int32)
            nv = np.ascontiguousarray(mask.sum(1) if nv is None else nv, np.int32)
            return lib.pllb_s2s_train_step_host(h, engine._np_ptr(i), engine._np_ptr(nv), engine._np_ptr(lab), B, Te, Td,
                                                mode, None)
        assert code() == 0
        bad = ids.copy(); bad[0, 1] = 300
        assert code(i=bad) == 1
        bad = labels.copy(); bad[0, 1] = 300
        assert code(lab=bad) == 1
        bad = labels.copy(); bad[0, 1] = -1
        assert code(lab=bad) == 1
        assert code(lab=np.full_like(labels, -100)) == 1
        assert code(nv=np.array([0, 3])) == 1 and code(nv=np.array([9, 3])) == 1
        assert code(mode=3) == 1
        big = np.zeros((3, 65), np.int32)
        assert code(i=big, lab=big, nv=np.ones(3), B=3, Te=65, Td=6) == 5       # TOO_LONG: above the position table
        assert code(i=big, lab=big, nv=np.ones(3), B=2, Te=6, Td=65) == 5
        assert code(i=big, lab=np.full((3, 7), 5), nv=np.ones(3), B=3, Te=8, Td=6) == 4   # OOM: above the capacity
        assert code(i=big, lab=np.full((3, 9), 5), nv=np.ones(3), B=2, Te=9, Td=6) == 4
        # the MLM and RescoreBert calls reject this handle
        loss = engine.ctypes.c_float()
        i32 = np.ascontiguousarray(ids, np.int32)
        assert lib.pllb_train_step_host(h, engine._np_ptr(i32), engine._np_ptr(np.ones(2, np.int32)),
                                        engine._np_ptr(i32), 2, 8, 2, engine.ctypes.byref(loss)) == 1
        p = engine._np_ptr(i32)
        assert lib.pllb_cls_train_step_host(h, p, p, p, p, p, p, 2, 8, 2, engine.ctypes.byref(loss), None) == 1
        # training takes operand_dtype 0 only
        import torch
        d = cfg.to_dict()
        s = engine.check_bart_config(d)
        sd_dev = {k: v.detach().float().cuda() for k, v in m.state_dict().items()}
        w, keep = engine.s2s_weights_struct(lambda k: sd_dev[k], d, 0)
        desc = _lib.S2sDesc(s["enc_layers"], s["dec_layers"], s["hidden"], s["num_heads"], s["enc_intermediate"],
                            s["dec_intermediate"], s["vocab"], s["max_position"], s["max_position"], 1e-5,
                            s["embed_scale"], CLS, SEP, 1)
        h2 = engine.ctypes.c_void_p()
        torch.cuda.synchronize()
        assert lib.pllb_s2s_train_create(engine.ctypes.byref(h2), engine.ctypes.byref(desc), engine.ctypes.byref(w),
                                         engine.ctypes.byref(tr._train_desc), 0) == 1
    # an s2s call rejects an MLM trainer
    bert_cfg = synth.BERT_TINY
    with engine.MlmTrainer(synth.random_init_state_dict(bert_cfg, 10), bert_cfg, device=0, max_rows=64, max_seq=16) as mt:
        i32 = np.ascontiguousarray(ids, np.int32)
        assert mt._lib.pllb_s2s_train_step_host(mt._h, engine._np_ptr(i32), engine._np_ptr(np.ones(2, np.int32)),
                                                engine._np_ptr(i32), 2, 8, 8, 2, None) == 1


def test_end_to_end_learns_a_permutation(tmp_path):
    """Random init, a fixed character permutation as the correction to learn; the device's epoch losses track the
    oracle trained on the same batches, and the exported model emits EOS and corrects held-out inputs."""
    import copy
    from asr_rescoring_b200.CorrectBart.model import CorrectBart, compute_cer
    from asr_rescoring_b200.CorrectBart.train import make_batches, train
    from asr_rescoring_b200.tokenizer import BertCharTokenizer
    chars = [chr(0x4E00 + 37 * i) for i in range(40)]
    vocab = ["[PAD]"] + [f"[unused{i}]" for i in range(99)] + ["[UNK]", "[CLS]", "[SEP]", "[MASK]"] + chars
    p = tmp_path / "vocab.txt"
    p.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    tok = BertCharTokenizer(str(p))
    perm = dict(zip(chars, np.random.default_rng(1).permutation(chars)))
    rng = np.random.default_rng(2)
    src = ["".join(rng.choice(chars, size=int(L))) for L in rng.integers(3, 9, size=544)]
    tgt = ["".join(perm[ch] for ch in s) for s in src]
    train_h, train_r, test_h, test_r = src[:512], tgt[:512], src[512:], tgt[512:]
    cfg = bo.bart_config(d_model=256, layers=2, ffn=1024, vocab=len(vocab), max_position=64, init_std=0.02)
    m = bo.make_model(cfg, seed=4, perturb=False)
    epochs, lr = 12, 1e-3
    sd, losses = train(m.state_dict(), cfg.to_dict(), tok, train_h, train_r, epochs=epochs, lr=lr, sents_per_batch=32,
                       dropout=0.0, attention_dropout=0.0)
    oracle = bto.train_epochs(copy.deepcopy(m), make_batches(tok, train_h, train_r, 32), epochs, lr)
    print(f"[e2e] device epoch losses {np.round(losses['train'], 4).tolist()}")
    print(f"[e2e] oracle epoch losses {np.round(oracle, 4).tolist()}")
    assert losses["train"][-1] < 0.5 * losses["train"][0]
    for d, o in zip(losses["train"], oracle):
        assert abs(d - o) <= 0.02 * o + 0.005          # measured: 0.0037 at a loss of 1.42
    model = CorrectBart(sd, cfg.to_dict(), tok, device=0, max_length=16)
    try:
        ids, lens = model.generate_packed(*_pack([tok.encode(t) for t in test_h]))
        preds = model.correct(test_h)
    finally:
        model.close()
    emitted = int((lens < 16).sum())
    cer = compute_cer(preds, test_r)
    print(f"[e2e] {emitted} of {len(test_h)} held-out sentences emit EOS before max_length; CER {cer:.4f}")
    assert emitted == len(test_h)
    assert cer < 0.05                                  # measured: 0


def _pack(sents):
    off = np.zeros(len(sents) + 1, np.int64)
    np.cumsum([len(s) for s in sents], out=off[1:])
    return np.array([t for s in sents for t in s], np.int32), off
