"""RescoreBert distillation on the GPU (engine.ClsTrainer, pllb_cls_train_*) against
oracle/rescorebert_train_oracle.py, the fp32 autograd restatement that pins the loss contract of
include/pllb.h (the reference's training script is not in the reference tree, so there is no
reference golden).

Tolerances (bf16 GEMM operands in forward, dgrad and wgrad; fp32 elsewhere): per-hypothesis scores
within 0.05 absolute (the bar of the scoring test); batch loss within 1 % relative plus 0.02; per-tensor
gradients within 6 % relative L2 error and cosine >= 0.998, as for the MLM trainer (the key bias, whose
true gradient is 0, is excepted the same way)."""
import ctypes

import numpy as np
import pytest
import torch

from asr_rescoring_b200 import _lib, cer_clients, engine, synth
from asr_rescoring_b200.RescoreBert import train as rb_train
from oracle import rescore_oracle
from oracle import rescorebert_train_oracle as rto

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("require_gpu")]
KEY_BIAS = "attention.self.key.bias"
POOLER = "bert.pooler."
LOSS_RTOL, LOSS_ATOL = 1e-2, 0.02
MWER = dict(md_weight=1.0, mwer_weight=1.0, am_weight=1.0)


def _nbest(cfg, n_utts, n_best, seed):
    """Synthetic N-best lists: token ids, AM scores, CER from the applied edit counts and a teacher-PLL stand-in."""
    nb = synth.make_nbest(n_utts, n_best, seed=seed)
    tok, off = nb.packed_tokens(cfg["vocab"])
    rng = np.random.default_rng(seed)
    tokens, pll, cer, i = {}, {}, {}, 0
    for u, (utt, hs) in enumerate(zip(nb.utt_ids, nb.hyps)):
        tokens[utt], pll[utt], cer[utt] = {}, {}, {}
        for k in range(len(hs)):
            h = f"hyp_{k + 1}"
            tokens[utt][h] = [int(t) for t in tok[off[i]:off[i + 1]]]
            pll[utt][h] = float(-2.0 * len(tokens[utt][h]) + rng.normal(0.0, 1.0))
            cer[utt][h] = float(nb.edits[u, k]) / len(nb.refs[u])
            i += 1
    return nb, tokens, pll, nb.hyps_score(), cer


def _trainer(sd, cfg, batches, **kw):
    rows, seq = rb_train.batch_capacity(batches)
    kw.setdefault("hidden_dropout", 0.0)
    kw.setdefault("attention_dropout", 0.0)
    return engine.ClsTrainer(sd, cfg, max_rows=rows, max_seq=seq, **kw)


def _step(tr, b, mode):
    return tr.step(b["input_ids"], b["attention_mask"], b["group"], b["target"], b["am"], b["err"], mode=mode)


@pytest.mark.parametrize("weights", [dict(md_weight=1.0, mwer_weight=0.0), MWER], ids=["md", "md_mwer"])
def test_batch_scores_loss_and_gradients_vs_oracle(weights):
    """Tiny shape, perturbed weights, dropout 0, rows of different lengths (padding inside the batch)."""
    cfg = synth.BERT_TINY
    sd = synth.random_rescorebert_state_dict(cfg, 21, perturb=True)
    _, tokens, pll, am, cer = _nbest(cfg, 4, 5, seed=3)
    b = rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=4)[0]
    assert (b["attention_mask"] == 0).any()
    o_loss, o_scores, o_grads = rto.loss_and_grads(sd, cfg, b, **weights)
    with _trainer(sd, cfg, [b], lr=1e-3, **weights) as tr:
        l0, s0 = _step(tr, b, 0)
        l2, s2 = _step(tr, b, 2)
        g = tr.grads()
    print(f"cls batch {weights}: loss oracle {o_loss:.5f}, eval {l0:.5f}, train {l2:.5f}; "
          f"max |ds| {np.abs(s0 - o_scores).max():.4f}")
    assert np.abs(s0 - o_scores).max() < 0.05 and np.array_equal(s0, s2) and l0 == l2
    assert abs(l0 - o_loss) <= LOSS_RTOL * abs(o_loss) + LOSS_ATOL
    assert set(g) == set(sd)
    worst = ("", 0.0, 1.0)
    for k, og in o_grads.items():
        d, og = g[k].double().reshape(og.shape), og.double()
        if k.endswith(KEY_BIAS):
            assert float(d.norm()) <= 1e-3 * float(o_grads[k.replace("key.bias", "query.bias")].norm()) + 1e-6, k
            continue
        rel = float((d - og).norm() / (og.norm() + 1e-30))
        cos = float((d * og).sum() / (d.norm() * og.norm() + 1e-30))
        if rel > worst[1]:
            worst = (k, rel, cos)
        assert rel <= 0.06 and cos >= 0.998, (k, rel, cos)
    print(f"gradients: worst tensor {worst[0]}: rel L2 error {worst[1]:.4f}, cosine {worst[2]:.5f}")
    assert not any(k.startswith(POOLER) for k in o_grads)
    assert all(float(g[k].abs().max()) == 0.0 for k in g if k.startswith(POOLER))
    assert float(g["bert.embeddings.word_embeddings.weight"][0].abs().max()) == 0.0      # padding_idx


def test_bert_base_twelve_layers_three_steps_vs_oracle():
    """bert-base-chinese shape and depth, random init, three AdamW steps at lr 1e-4 (MD + MWER) on one batch
    of two 10-best lists: the losses follow the fp32 autograd oracle and fall."""
    cfg = synth.BERT_BASE_CHINESE
    sd = synth.random_rescorebert_state_dict(cfg, 10)
    _, tokens, pll, am, cer = _nbest(cfg, 2, 10, seed=11)
    b = rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=2)[0]
    o_losses = rto.run_steps(rto.parameters(sd), cfg, [b] * 3, 1e-4, **MWER)
    with _trainer(sd, cfg, [b], lr=1e-4, **MWER) as tr:
        tr.reset_optimizer(1e-4)
        got = [_step(tr, b, 1)[0] for _ in range(3)]
    print(f"bert-base-chinese, 12 layers: device losses {[round(x, 4) for x in got]}, oracle {[round(x, 4) for x in o_losses]}")
    assert all(abs(a - o) <= LOSS_RTOL * abs(o) + LOSS_ATOL for a, o in zip(got, o_losses))
    assert got[2] < got[1] < got[0]


def test_steps_are_deterministic_and_graph_replays_match_eager(monkeypatch):
    cfg = synth.BERT_TINY
    sd = synth.random_rescorebert_state_dict(cfg, 5, perturb=True)
    _, tokens, pll, am, cer = _nbest(cfg, 6, 4, seed=9)
    b1, b2 = rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=3)
    assert b1["input_ids"].shape != b2["input_ids"].shape
    # every forward pass draws new dropout masks, so repeated passes are compared at dropout 0
    with _trainer(sd, cfg, [b1, b2], **MWER) as tr:
        la, sa = _step(tr, b1, 2)
        ga = tr.grads()
        lb, sb = _step(tr, b1, 2)
        gb = tr.grads()
    assert la == lb and np.array_equal(sa, sb) and all(bool((ga[k] == gb[k]).all()) for k in ga)

    def run():
        with _trainer(sd, cfg, [b1, b2], lr=1e-3, hidden_dropout=0.1, attention_dropout=0.1, seed=5, **MWER) as tr:
            out = [_step(tr, b1, 1) for _ in range(5)] + [_step(tr, b2, 1) for _ in range(3)]
            out += [_step(tr, b1, 0) for _ in range(3)]
            return [o[0] for o in out], [o[1] for o in out], tr.state_dict(), tr.graph_replays(), tr.kernel_launches()

    l_g, s_g, sd_g, replays, launches_g = run()
    monkeypatch.setenv("PLLB_TRAIN_GRAPH", "0")
    l_e, s_e, sd_e, replays_e, launches_e = run()
    print(f"graph: {replays} replays, {launches_g} launches in 11 steps")
    assert replays == 4 + 2 + 2 and replays_e == 0 and launches_g == launches_e
    assert l_g == l_e and all(np.array_equal(a, b) for a, b in zip(s_g, s_e))
    assert all(bool((sd_g[k] == sd_e[k]).all()) for k in sd_g)
    assert len(set(l_g[:5])) == 5


def test_distillation_end_to_end_round_trip(tmp_path):
    """Teacher PLLs from PllScorer, CERs from cer_clients.hyps_cer, a few epochs of RescoreBert/train.py (dropout
    0.1): the loss falls; the exported state_dict scores through RescoreBert like the trainer's eval pass, keeps
    the pooler bit for bit, and its scores go through rescore.find_best_weight."""
    from asr_rescoring_b200 import rescore
    from asr_rescoring_b200.RescoreBert.model import RescoreBert
    cfg = synth.BERT_TINY
    teacher = synth.random_init_state_dict(cfg, 4, perturb=True)
    student = synth.random_rescorebert_state_dict(cfg, 7)
    nb = synth.make_nbest(12, 4, seed=2)
    tok, off = nb.packed_tokens(cfg["vocab"])
    tokens = {u: {f"hyp_{k + 1}": [int(t) for t in tok[off[i * 4 + k]:off[i * 4 + k + 1]]] for k in range(4)}
              for i, u in enumerate(nb.utt_ids)}
    with engine.PllScorer(teacher, cfg) as sc:
        pll = sc.score_hyps(tokens)
    cer = cer_clients.hyps_cer(nb.hyps_text(), nb.ref_text())
    am = nb.hyps_score()
    sd, losses = rb_train.train(student, tokens, pll, am, cer, epochs=4, lr=1e-3, utts_per_batch=4, seed=1, **MWER)
    print(f"distillation epoch losses {[round(x, 3) for x in losses['train']]}")
    assert losses["train"][-1] < losses["train"][0]
    assert set(sd) == set(student)
    assert all(torch.equal(sd[k], student[k]) for k in student if k.startswith(POOLER))
    assert not torch.equal(sd["linear.weight"], student["linear.weight"])
    batches = rb_train.make_batches(tokens, pll, am, cer, 4)
    ev = {}
    with _trainer(sd, cfg, batches, **MWER) as tr:
        rb_train.run_one_epoch(tr, batches, False, scores=ev)
    with RescoreBert(sd, cfg) as m:
        got = m.score_hyps(tokens)
    worst = max(abs(got[u][h] - ev[u][h]) for u in tokens for h in tokens[u])
    print(f"exported student: max |RescoreBert score - trainer eval score| {worst:.4f}")
    assert worst < 0.05
    lm = [[got[u][h] for h in tokens[u]] for u in tokens]
    bw, bc = rescore.find_best_weight(nb.am.tolist(), lm, nb.hyps, nb.refs, rescore_oracle.config(4))
    assert 0.0 <= bw <= 1.0 and np.isfinite(bc)


def test_invalid_inputs_cross_kind_calls_and_workspace():
    cfg = synth.BERT_TINY
    sd = synth.random_rescorebert_state_dict(cfg, 2)
    _, tokens, pll, am, cer = _nbest(cfg, 2, 3, seed=4)
    b = rb_train.make_batches(tokens, pll, am, cer, utts_per_batch=2)[0]
    args = lambda **o: [o.get(k, b[k]) for k in ("input_ids", "attention_mask", "group", "target", "am", "err")]  # noqa: E731
    oov = b["input_ids"].copy()
    oov[0, 1] = cfg["vocab"]
    with _trainer(sd, cfg, [b], **MWER) as tr:
        for bad in (dict(group=np.array([1, 1, 1, 2, 2, 2])), dict(group=np.array([0, 0, 1, 0, 1, 1])),
                    dict(group=np.array([0, 0, 0, 2, 2, 2])), dict(target=np.where(np.arange(6) == 2, np.nan, b["target"])),
                    dict(am=np.full(6, np.inf)), dict(input_ids=oov)):
            with pytest.raises(_lib.PllbError) as e:
                tr.step(*args(**bad), mode=0)
            assert e.value.code == 1, bad
        hole = b["attention_mask"].copy()
        hole[0, 1] = 0
        with pytest.raises(ValueError):
            tr.step(*args(attention_mask=hole), mode=0)
        wide = np.pad(b["input_ids"], ((0, 0), (0, 1)))
        with pytest.raises(_lib.PllbError) as e:
            tr.step(*args(input_ids=wide, attention_mask=np.pad(b["attention_mask"], ((0, 0), (0, 1)))), mode=0)
        assert e.value.code == 5                                 # T > max_seq
        big = {k: np.concatenate([b[k], b[k]]) for k in ("input_ids", "attention_mask", "target", "am", "err")}
        with pytest.raises(_lib.PllbError) as e:
            tr.step(*args(group=np.repeat([0, 1, 2, 3], 3), **big), mode=0)
        assert e.value.code == 4                                 # B * T > max_rows
        # a group of one hypothesis: P = 1, so MWER adds nothing (the loss is the MD term)
        single = dict(group=np.array([0, 0, 0, 1, 2, 3]))
        l_md, s = tr.step(*args(**single), mode=0)
        exp = float(rto.losses(torch.tensor(s, dtype=torch.float64), b["target"], b["am"], b["err"], single["group"], **MWER)[0])
        assert abs(l_md - exp) <= 1e-4 * abs(exp)
        # cross-kind calls
        lib, h = tr._lib, tr._h
        n = b["input_ids"].size
        i32 = np.zeros(n, np.int32)
        loss = ctypes.c_float(0.0)
        rc = lib.pllb_train_step_host(h, i32.ctypes.data, i32.ctypes.data, i32.ctypes.data, 1, 1, 0, ctypes.byref(loss))
        assert rc == 1
        assert lib.pllb_train_row_losses_host(h, np.zeros(1, np.float32).ctypes.data, 1) == 1
        w = _lib.Weights()
        layers = (_lib.LayerWeights * cfg["num_layers"])()
        w.layers = ctypes.cast(layers, ctypes.POINTER(_lib.LayerWeights))
        assert lib.pllb_train_export(h, ctypes.byref(w)) == 1 and lib.pllb_train_export_grads(h, ctypes.byref(w)) == 1
        cls_ws = tr.workspace_bytes()
    mlm_sd = synth.random_init_state_dict(cfg, 2)
    rows, seq = rb_train.batch_capacity([b])
    with engine.MlmTrainer(mlm_sd, cfg, max_rows=rows, max_seq=seq) as mt:
        f = np.zeros(1, np.float32)
        assert mt._lib.pllb_cls_train_step_host(mt._h, i32.ctypes.data, i32.ctypes.data, i32.ctypes.data, f.ctypes.data,
                                                f.ctypes.data, f.ctypes.data, 1, 1, 0, ctypes.byref(loss), None) == 1
        assert mt._lib.pllb_cls_train_export(mt._h, ctypes.byref(w), None, None) == 1
        assert mt._lib.pllb_cls_train_export_grads(mt._h, ctypes.byref(w), None, None) == 1
    # memory at the bert-base-chinese vocabulary: the MLM trainer's [R, Vp] logits (fp32) and their gradient (bf16)
    # and the two bf16 decoder copies are absent from a CLS trainer of the same capacity
    big_cfg = dict(synth.BERT_BASE_CHINESE, num_layers=1)
    R, T, Vp, H = 1024, 64, 21248, 768
    with engine.ClsTrainer(synth.random_rescorebert_state_dict(big_cfg, 1), big_cfg, max_rows=R, max_seq=T) as ct:
        cls_big = ct.workspace_bytes()
    with engine.MlmTrainer(synth.random_init_state_dict(big_cfg, 1), big_cfg, max_rows=R, max_seq=T) as mt:
        mlm_big = int(mt._lib.pllb_train_workspace_bytes(mt._h))
    print(f"workspace, bert-base vocabulary, 1 layer, {R} rows: CLS {cls_big / 1e6:.0f} MB, MLM {mlm_big / 1e6:.0f} MB; "
          f"tiny: CLS {cls_ws / 1e6:.1f} MB")
    assert mlm_big - cls_big >= R * Vp * 6 + 2 * Vp * H * 2
