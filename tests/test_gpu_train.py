"""MLM fine-tuning on the GPU (SURVEY.md §8f rank 4; reference MLM_PLL/main.py:73-99,117-161) against
oracle/train_oracle.py (autograd restatement, pinned to the unmodified reference loop by
tests/golden/train_golden.json).  Everything goes through the C ABI (pllb_train_*).

Tolerances (bf16 GEMM operands in forward, dgrad and wgrad; fp32 everything else): batch loss within
0.02 nats; per-tensor gradients within 6 % relative L2 error and cosine >= 0.998; the AdamW update
itself (given the device's own gradients) within 2e-7 absolute; epoch losses of the golden runs
within 0.05."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from asr_rescoring_b200 import engine, synth
from oracle import pll_oracle, train_oracle

pytestmark = [pytest.mark.gpu, pytest.mark.usefixtures("require_gpu")]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEY_BIAS = "attention.self.key.bias"      # true gradient 0 (softmax ignores a per-row constant): noise on both sides


def _case(gold_dir, name):
    gold = json.load(open(os.path.join(gold_dir, "train_golden.json")))
    case = next(c for c in gold["cases"] if c["name"] == name)
    sd = synth.random_init_state_dict(case["cfg"], case["seed"], case["perturb"])
    return case, sd, train_oracle.training_rows(case["train_tokens"]), train_oracle.training_rows(case["dev_tokens"])


def _batch(rows):
    ids, am, lab, *_ = pll_oracle.collate(rows)
    return ids.numpy().astype(np.int32), am.numpy().astype(np.int32), lab.numpy().astype(np.int32)


def test_batch_loss_and_gradients_vs_oracle(gold_dir):
    """One zero-padded batch (rows of different lengths, so pad positions with label 0 are inside):
    loss in eval mode and in train mode without dropout, and every parameter gradient."""
    case, sd, rows, _ = _case(gold_dir, "tiny_perturbed")
    cfg = case["cfg"]
    batch = rows[3:35]                                  # spans three sentences of different lengths
    ids, am, lab = _batch(batch)
    assert (am == 0).any()
    o_loss, o_grads = train_oracle.loss_and_grads(sd, cfg, batch)
    with engine.MlmTrainer(sd, cfg, lr=1e-3, hidden_dropout=0.0, attention_dropout=0.0, max_rows=ids.size, max_seq=ids.shape[1]) as tr:
        l0 = tr.step(ids, am, lab, mode=0)
        l2 = tr.step(ids, am, lab, mode=2)
        g = tr.grads()
        g_again = (tr.step(ids, am, lab, mode=2), tr.grads())
        launches = tr.kernel_launches()
    print(f"train batch: loss oracle {o_loss:.5f}, device eval {l0:.5f}, train {l2:.5f}; {launches} kernel launches in 3 passes")
    assert abs(l0 - o_loss) <= 0.02 and l0 == l2 and launches > 100
    worst = ("", 0.0, 1.0)
    for k, og in o_grads.items():
        d = g[k].double()
        og = og.double()
        if k.endswith(KEY_BIAS):
            assert float(d.norm()) <= 1e-3 * float(o_grads[k.replace("key.bias", "query.bias")].norm()) + 1e-6, k
            continue
        rel = float((d - og).norm() / (og.norm() + 1e-30))
        cos = float((d * og).sum() / (d.norm() * og.norm() + 1e-30))
        if rel > worst[1]:
            worst = (k, rel, cos)
        assert rel <= 0.06 and cos >= 0.998, (k, rel, cos)
    print(f"gradients: worst tensor {worst[0]}: rel L2 error {worst[1]:.4f}, cosine {worst[2]:.5f}")
    # tied entries come back as one tensor; determinism: a second identical pass is bit-identical
    assert g["cls.predictions.decoder.weight"] is g["bert.embeddings.word_embeddings.weight"]
    assert g_again[0] == l2 and all(bool((g_again[1][k] == g[k]).all()) for k in g if not k.endswith("position_ids"))
    # nn.Embedding(padding_idx=0): the lookup sends nothing to row 0, the tied decoder does
    assert float(g["bert.embeddings.word_embeddings.weight"][0].abs().sum()) > 0


def test_bert_base_shape_two_layers_vs_oracle():
    """H = 768 / 12 heads / I = 3072 / vocab 21128 (not a multiple of the 256-column vocab tile): the shape
    the reference fine-tunes (train.yaml:23-24), two layers deep so the CPU oracle stays cheap."""
    cfg = dict(synth.BERT_BASE_CHINESE, num_layers=2)
    sd = synth.random_init_state_dict(cfg, 10, perturb=True)
    nb = synth.make_nbest(5, 1, seed=7)
    tok, off = nb.packed_tokens()
    rows = train_oracle.training_rows([[int(t) for t in tok[off[i]:off[i + 1]]] for i in range(len(off) - 1)])[5:37]
    ids, am, lab = _batch(rows)
    o_loss, o_grads = train_oracle.loss_and_grads(sd, cfg, rows)
    with engine.MlmTrainer(sd, cfg, hidden_dropout=0.0, attention_dropout=0.0, max_rows=ids.size, max_seq=ids.shape[1]) as tr:
        loss = tr.step(ids, am, lab, mode=2)
        g = tr.grads()
    assert abs(loss - o_loss) <= 0.02, (loss, o_loss)
    worst = 0.0
    for k, og in o_grads.items():
        if k.endswith(KEY_BIAS):
            continue
        d, og = g[k].double(), og.double()
        rel = float((d - og).norm() / (og.norm() + 1e-30))
        worst = max(worst, rel)
        assert rel <= 0.06, (k, rel)
    print(f"bert-base shape, 2 layers: loss {loss:.5f} (oracle {o_loss:.5f}), worst gradient rel L2 error {worst:.4f}")


def test_bert_base_twelve_layers_three_steps_vs_oracle():
    """The shape and depth the reference fine-tunes (bert-base-chinese, train.yaml:23-24), three AdamW steps at
    lr 1e-4 on batches of 32 rows: the batch losses follow the fp32 autograd oracle within 0.02 nats, and the
    loss falls."""
    cfg = synth.BERT_BASE_CHINESE
    sd = synth.random_init_state_dict(cfg, 10)
    nb = synth.make_nbest(8, 1, seed=11)
    tok, off = nb.packed_tokens()
    rows = train_oracle.training_rows([[int(t) for t in tok[off[i]:off[i + 1]]] for i in range(len(off) - 1)])
    assert len(rows) >= 96
    params = train_oracle.parameters(sd)
    o_losses = []
    train_oracle.run_one_epoch(params, cfg, rows[:96], 32, 1e-4, True, batch_losses=o_losses)
    got = []
    with engine.MlmTrainer(sd, cfg, lr=1e-4, hidden_dropout=0.0, attention_dropout=0.0, max_rows=32 * 40, max_seq=40) as tr:
        tr.reset_optimizer(1e-4)
        for s0 in (0, 32, 64):
            got.append(tr.step(*_batch(rows[s0:s0 + 32]), mode=1))
    print(f"bert-base-chinese, 12 layers: device losses {[round(x, 4) for x in got]}, oracle {[round(x, 4) for x in o_losses]}")
    assert all(abs(a - b) <= 0.02 for a, b in zip(got, o_losses)) and got[2] < got[0]


def test_adamw_update_matches_torch_given_the_same_gradients(gold_dir):
    """The optimizer in isolation: gradients of a mode-2 pass, then a mode-1 pass on the same batch
    (same gradients: no dropout, deterministic kernels); torch.optim.AdamW on CPU fed with the
    device's gradients must land on the device's new weights.  Two steps, so the moments matter."""
    import torch
    case, sd, rows, _ = _case(gold_dir, "tiny_perturbed")
    cfg, lr = case["cfg"], 1e-3
    with engine.MlmTrainer(sd, cfg, lr=lr, hidden_dropout=0.0, attention_dropout=0.0, max_rows=2048, max_seq=64) as tr:
        tr.reset_optimizer(lr)
        params = {k: v.clone().float().requires_grad_(True) for k, v in sd.items()
                  if k not in train_oracle.TIED and not k.endswith("position_ids")}
        opt = torch.optim.AdamW(list(params.values()), lr=lr)
        for s0 in (0, 32):
            ids, am, lab = _batch(rows[s0:s0 + 32])
            tr.step(ids, am, lab, mode=2)
            g = tr.grads()
            tr.step(ids, am, lab, mode=1)
            for k, p in params.items():
                p.grad = g[k].clone()
            opt.step()
            new = tr.state_dict()
            worst = max(float((new[k] - p.detach()).abs().max()) for k, p in params.items())
            print(f"AdamW step from row {s0}: max |device - torch| = {worst:.2e}")
            assert worst <= 2e-7
        assert new["cls.predictions.decoder.weight"] is new["bert.embeddings.word_embeddings.weight"]
        # token_type row 1 never gets a gradient but is still decayed (weight_decay on every parameter)
        tt0, tt1 = sd["bert.embeddings.token_type_embeddings.weight"][1], new["bert.embeddings.token_type_embeddings.weight"][1]
        assert torch.allclose(tt1, tt0 * (1 - lr * 0.01) ** 2, rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("name", ["tiny_lr1e-5", "tiny_perturbed"])
def test_drop_in_epochs_match_the_reference_golden(gold_dir, name):
    """The drop-in run_one_epoch (train pass with a fresh AdamW per epoch, then the dev-loss pass)
    against the epoch losses the UNMODIFIED reference loop returned (tests/golden/train_golden.json)."""
    import importlib
    m = importlib.import_module("asr_rescoring_b200.MLM_PLL.main")
    case, sd, train_rows, dev_rows = _case(gold_dir, name)
    conf = SimpleNamespace(lr=case["lr"], device="cuda:0")
    dl = SimpleNamespace(shuffle=False, batch_size=case["batch_size"], num_worker=0)
    train_loader = m.set_dataloader(dl, m.MyDataset(train_rows), False)
    dev_loader = m.set_dataloader(dl, m.MyDataset(dev_rows), True)
    longest = max(len(r["input_ids"]) for r in train_rows + dev_rows)
    with engine.MlmTrainer(sd, case["cfg"], lr=case["lr"], hidden_dropout=0.0, attention_dropout=0.0,
                           max_rows=case["batch_size"] * longest, max_seq=longest) as tr:
        for e in range(case["epochs"]):
            tl = m.run_one_epoch(config=conf, model=tr, dataloader=train_loader, output_score=None, train_mode=True, do_scoring=False)
            dv = m.run_one_epoch(config=conf, model=tr, dataloader=dev_loader, output_score=None, train_mode=False, do_scoring=False)
            print(f"{name} epoch {e + 1}: train {tl:.4f} (reference {case['train_loss'][e]:.4f}), dev {dv:.4f} ({case['dev_loss'][e]:.4f})")
            assert abs(tl - case["train_loss"][e]) <= 0.05 and abs(dv - case["dev_loss"][e]) <= 0.05
        final = tr.state_dict()
    # direction of travel of the large tensors agrees with the reference run (summaries in the golden)
    import torch
    for k in ("bert.encoder.layer.0.intermediate.dense.weight", "cls.predictions.transform.dense.weight"):
        ref = case["final_minus_init"][k]
        delta = (final[k] - sd[k]).double().reshape(-1)
        gsign = torch.Generator().manual_seed(1234 + delta.numel() % 977)
        sign = torch.randint(0, 2, (delta.numel(),), generator=gsign, dtype=torch.int64).double() * 2 - 1
        assert abs(float(delta.norm()) - ref["norm"]) <= 0.1 * ref["norm"], (k, float(delta.norm()), ref["norm"])
        assert abs(float((delta * sign).sum()) - ref["proj"]) <= 0.25 * ref["norm"], k


def test_dropout_is_seeded_and_eval_ignores_it(gold_dir):
    case, sd, rows, _ = _case(gold_dir, "tiny_perturbed")
    cfg = case["cfg"]
    ids, am, lab = _batch(rows[:32])

    def run(seed, p):
        with engine.MlmTrainer(sd, cfg, lr=1e-4, hidden_dropout=p, attention_dropout=p, seed=seed, max_rows=2048, max_seq=64) as tr:
            ev = tr.step(ids, am, lab, mode=0)
            return ev, [tr.step(ids, am, lab, mode=1) for _ in range(3)], tr.state_dict()

    ev0, l0, _ = run(1, 0.0)
    ev_a, la, sa = run(1, 0.1)
    ev_b, lb, sb = run(1, 0.1)
    ev_c, lc, _ = run(2, 0.1)
    assert ev0 == ev_a == ev_c                                   # model.eval(): dropout off
    assert la == lb and all(bool((sa[k] == sb[k]).all()) for k in sa)          # same seed: bit-identical training
    assert la != lc and la != l0 and np.isfinite(la).all()
    assert abs(la[0] - l0[0]) < 0.5 and la[0] != la[1]           # a perturbation, and a new mask every step
    # heavy dropout still trains finitely (inverse-keep scaling in forward and backward)
    _, lh, _ = run(3, 0.5)
    assert np.isfinite(lh).all()


def test_graph_replay_is_bit_identical_to_eager_launches(gold_dir, monkeypatch):
    """A batch shape runs eagerly once, is captured as a CUDA graph on its second occurrence and replayed
    afterwards (dropout seed and Adam bias corrections are read from device memory, so the graph is
    step-independent).  Same losses and same final weights, bit for bit, as with PLLB_TRAIN_GRAPH=0."""
    case, sd, rows, _ = _case(gold_dir, "tiny_perturbed")
    ids, am, lab = _batch(rows[:32])
    ids2, am2, lab2 = _batch(rows[40:56])

    def run():
        with engine.MlmTrainer(sd, case["cfg"], lr=1e-3, hidden_dropout=0.1, attention_dropout=0.1, seed=5, max_rows=2048, max_seq=64) as tr:
            losses = [tr.step(ids, am, lab, mode=1) for _ in range(5)]
            losses += [tr.step(ids2, am2, lab2, mode=1) for _ in range(3)] + [tr.step(ids, am, lab, mode=0) for _ in range(3)]
            return losses, tr.state_dict(), tr.graph_replays(), tr.kernel_launches()

    l_graph, s_graph, replays, launches_g = run()
    monkeypatch.setenv("PLLB_TRAIN_GRAPH", "0")
    l_eager, s_eager, replays_e, launches_e = run()
    assert replays == 4 + 2 + 2 and replays_e == 0 and launches_g == launches_e
    assert l_graph == l_eager and all(bool((s_graph[k] == s_eager[k]).all()) for k in s_graph)
    assert len(set(l_graph[:5])) == 5                 # a new dropout mask and a new Adam step every replay


def test_fine_tuned_checkpoint_is_scored_by_the_scoring_path(gold_dir, tmp_path):
    """task: training through the CLI (MLM_PLL/main.py:117-161 drop-in) -> checkpoint_<epoch>.pth + loss.json;
    the checkpoint is a bare state_dict that the scoring path loads (MLM_PLL/main.py:185-187) and whose PLLs
    match the fp32 oracle on the SAME fine-tuned weights."""
    import torch
    case, sd, train_rows, dev_rows = _case(gold_dir, "tiny_lr1e-5")
    (tmp_path / "out").mkdir()
    json.dump(train_rows, open(tmp_path / "train.json", "w"))
    json.dump(dev_rows, open(tmp_path / "dev.json", "w"))
    torch.save(sd, tmp_path / "start.pth")
    (tmp_path / "train.yaml").write_text(f"""
task: training
seed: 10
lr: 0.0005
epoch: 2
device: "cuda:0"
train_data_path: "{tmp_path}/train.json"
dev_data_path: "{tmp_path}/dev.json"
output_path: "{tmp_path}/out"
num_of_data: 99999999
dataloader:
  shuffle: True
  batch_size: 32
  num_worker: 5
model:
  bert: "bert-tiny-test"
  pretrained_path: "{tmp_path}/start.pth"
resume:
  start_from:
  checkpoint_path:
""")
    script = os.path.join(ROOT, "asr-rescoring_b200", "MLM_PLL", "main.py")
    out = subprocess.run([sys.executable, script, "--config", str(tmp_path / "train.yaml")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-2000:]
    loss = json.load(open(tmp_path / "out" / "loss.json"))
    assert len(loss["train"]) == 2 and len(loss["dev"]) == 2 and loss["train"][1] < loss["train"][0] and loss["dev"][1] < loss["dev"][0]
    ck = torch.load(tmp_path / "out" / "checkpoint_2.pth", map_location="cpu")
    assert set(ck.keys()) == set(sd.keys()) and not torch.equal(ck["cls.predictions.bias"], sd["cls.predictions.bias"])
    assert ck["cls.predictions.decoder.weight"].data_ptr() == ck["bert.embeddings.word_embeddings.weight"].data_ptr()
    hyps = {"u": {f"hyp_{i + 1}": t for i, t in enumerate(case["dev_tokens"])}}
    with engine.PllScorer(ck, case["cfg"]) as sc:
        got = sc.score_hyps(hyps)
    exp = pll_oracle.score_hyps(ck, case["cfg"], hyps)
    before = pll_oracle.score_hyps(sd, case["cfg"], hyps)
    worst = max(abs(got["u"][h] - exp["u"][h]) for h in exp["u"])
    moved = max(abs(before["u"][h] - exp["u"][h]) for h in exp["u"])
    print(f"fine-tuned checkpoint: max |dPLL| vs oracle {worst:.4f}; fine-tuning moved the PLLs by up to {moved:.2f} nats")
    assert worst <= 0.05 and moved > 0.2


def test_scoring_through_the_trainer_matches_the_scoring_path(gold_dir):
    """run_one_epoch(do_scoring=True) on a trainer — the padded-batch forward of the training path, row by row as
    the reference does it (MLM_PLL/main.py:100-107) — gives the PLLs of the varlen scoring path and of the oracle;
    with train_mode=True as well (dropout 0) the scores are those of the weights BEFORE each batch's update."""
    import importlib
    m = importlib.import_module("asr_rescoring_b200.MLM_PLL.main")
    case, sd, _, _ = _case(gold_dir, "tiny_lr1e-5")
    hyps = {"u1": {"hyp_1": case["dev_tokens"][0], "hyp_2": case["dev_tokens"][1]}, "u2": {"hyp_1": case["dev_tokens"][2]}}
    rows = [r for u, hs in hyps.items() for h, t in hs.items() for r in pll_oracle.expand_rows(t, u, h)]
    skel = lambda: {u: {h: 0 for h in hs} for u, hs in hyps.items()}
    exp = pll_oracle.score_hyps(sd, case["cfg"], hyps)
    conf = SimpleNamespace(lr=1e-5, device="cuda:0")
    loader = m.set_dataloader(SimpleNamespace(shuffle=False, batch_size=32, num_worker=0), m.MyDataset(rows), True)
    longest = max(len(r["input_ids"]) for r in rows)
    with engine.MlmTrainer(sd, case["cfg"], lr=1e-5, hidden_dropout=0.0, attention_dropout=0.0, max_rows=32 * longest, max_seq=longest) as tr:
        got = m.run_one_epoch(config=conf, model=tr, dataloader=loader, output_score=skel(), train_mode=False, do_scoring=True)
        got_tr = m.run_one_epoch(config=conf, model=tr, dataloader=loader, output_score=skel(), train_mode=True, do_scoring=True)
    with engine.PllScorer(sd, case["cfg"]) as sc:
        fast = sc.score_hyps(hyps)
    for u in hyps:
        for h in hyps[u]:
            assert abs(got[u][h] - exp[u][h]) <= 0.05 and abs(got[u][h] - fast[u][h]) <= 0.05, (u, h, got[u][h], exp[u][h], fast[u][h])
            assert abs(got_tr[u][h] - exp[u][h]) <= 0.3          # lr 1e-5: the weights move a little between batches


@pytest.mark.parametrize("kind", ["mlm", "cls"])
def test_state_dict_round_trips_through_the_flat_buffers(gold_dir, kind):
    """Import and export walk the same tensor list: right after construction state_dict() is the given fp32
    state_dict bit for bit (tied decoder and pass-through entries included), the gradients of a step come back
    under the same keys, and a null encoder pointer is rejected by the create call."""
    import ctypes
    import torch
    from asr_rescoring_b200 import _lib
    case, sd, rows, _ = _case(gold_dir, "tiny_perturbed")
    cfg = case["cfg"]
    ids, am, lab = _batch(rows[:8])
    B = ids.shape[0]
    kw = dict(hidden_dropout=0.0, attention_dropout=0.0, max_rows=ids.size, max_seq=ids.shape[1])
    if kind == "mlm":
        tr = engine.MlmTrainer(sd, cfg, **kw)
        step = lambda: tr.step(ids, am, lab, mode=2)                                  # noqa: E731
        create = lambda h, w: tr._lib.pllb_train_create(ctypes.byref(h), ctypes.byref(tr._desc), ctypes.byref(w),  # noqa: E731
                                                        ctypes.byref(tr._train_desc), 0)
    else:
        sd = synth.random_rescorebert_state_dict(cfg, 3, perturb=True)
        tr = engine.ClsTrainer(sd, cfg, mwer_weight=1.0, **kw)
        grp = (np.arange(B) * 2 // B).astype(np.int32)
        vals = [np.linspace(-1.0, 1.0, B, dtype=np.float32) * s for s in (30.0, 10.0, 0.2)]
        step = lambda: tr.step(ids, am, grp, *vals, mode=2)[0]                        # noqa: E731
        lin = [sd[k].cuda().reshape(-1) for k in ("linear.weight", "linear.bias")]
        ld = _lib.ClsLossDesc(1.0, 1.0, 1.0)
        create = lambda h, w: tr._lib.pllb_cls_train_create(  # noqa: E731
            ctypes.byref(h), ctypes.byref(tr._desc), ctypes.byref(w), ctypes.c_void_p(lin[0].data_ptr()),
            ctypes.c_void_p(lin[1].data_ptr()), ctypes.byref(tr._train_desc), ctypes.byref(ld), 0)
    bits = lambda t: t.contiguous().reshape(-1).view(torch.uint8)                     # noqa: E731
    with tr:
        got = tr.state_dict()
        assert list(got) == list(sd)
        for k, v in sd.items():
            assert got[k].dtype == v.dtype and got[k].shape == v.shape and torch.equal(bits(got[k]), bits(v)), k
        if kind == "mlm":
            assert got["cls.predictions.decoder.weight"] is got["bert.embeddings.word_embeddings.weight"]
            assert got["cls.predictions.decoder.bias"] is got["cls.predictions.bias"]
        else:
            assert all(got[k] is v for k, v in sd.items() if k.startswith("bert.pooler."))
        assert np.isfinite(step())
        g = tr.grads()
        assert list(g) == list(sd) and all(bool(torch.isfinite(v).all()) for v in g.values())
        w, keep = tr._weights_in(sd)
        w.layers[cfg["num_layers"] - 1].out_ln_b = None
        h = ctypes.c_void_p()
        assert create(h, w) == 1 and not h.value
        assert b"null" in tr._lib.pllb_last_error()
        del keep


def test_training_argument_errors(gold_dir):
    case, sd, rows, _ = _case(gold_dir, "tiny_lr1e-5")
    ids, am, lab = _batch(rows[:8])
    from asr_rescoring_b200._lib import PllbError
    with engine.MlmTrainer(sd, case["cfg"], hidden_dropout=0.0, attention_dropout=0.0, max_rows=ids.size, max_seq=ids.shape[1]) as tr:
        bad = ids.copy(); bad[0, 1] = case["cfg"]["vocab"]
        with pytest.raises(PllbError):                          # IndexError in the reference's embedding lookup
            tr.step(bad, am, lab, mode=0)
        hole = am.copy(); hole[0, 1] = 0
        with pytest.raises(ValueError):                         # only collate's prefix masks are supported
            tr.step(ids, hole, lab, mode=0)
        wide = np.zeros((1, ids.shape[1] + 1), np.int32)
        with pytest.raises(PllbError) as e:
            tr.step(wide, np.ones_like(wide), wide, mode=0)
        assert e.value.code == 5                                # PLLB_ERR_TOO_LONG
        big = np.tile(ids, (2, 1))
        with pytest.raises(PllbError) as e:
            tr.step(big, np.tile(am, (2, 1)), np.tile(lab, (2, 1)), mode=0)
        assert e.value.code == 4                                # PLLB_ERR_OOM: more rows than max_rows
        assert np.isfinite(tr.step(ids, am, lab, mode=0))
    with pytest.raises(ValueError):
        engine.MlmTrainer({k: v for k, v in sd.items() if not k.startswith("cls.")}, case["cfg"])
