"""RescoreBert distillation: train the [CLS] -> Linear(H, 1) student on the teacher's PLLs.

The teacher scores come from ``MLM_PLL/main.py`` (``train_lm.json``: {utt: {hyp: PLL}}), the AM scores
from ``hyps_score.json`` and the per-hypothesis CERs from ``hyps_cer.json`` (or
``cer_clients.hyps_cer``).  Batches hold whole utterances, in input order; the hypotheses of an
utterance are contiguous rows and form one group of the MWER loss.  The step runs in
``engine.ClsTrainer`` (include/pllb.h, ``pllb_cls_train_*``, states the losses):

    from asr_rescoring_b200.RescoreBert.train import train
    from asr_rescoring_b200.RescoreBert.model import RescoreBert
    sd, losses = train(student_sd, tokens, pll, am, cer, epochs=3, lr=1e-5, mwer_weight=1.0)
    with RescoreBert(sd) as m:
        lm = m.score_hyps(dev_tokens)          # dev_lm.json for rescore.py

``tokens`` is {utt: {hyp: wordpiece ids}} without [CLS] / [SEP]; the other three dicts have the
same keys.  There is no YAML front end: the reference's training configuration is not part of the
reference tree, so the driver takes plain arguments.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from ..engine import ClsTrainer

Scores = Dict[str, Dict[str, float]]


def make_batches(tokens: Dict[str, Dict[str, Sequence[int]]], pll: Scores, am: Scores, cer: Scores,
                 utts_per_batch: int, cls_id: int = 101, sep_id: int = 102) -> List[dict]:
    """Padded batches of ``utts_per_batch`` whole utterances in input order.  Each batch is a dict of
    input_ids / attention_mask int32 [B, T] ([CLS] t [SEP], right zero padding), group int32 [B]
    (0-based utterance index within the batch), target / am / err float32 [B], and the (utt, hyp)
    key of every row."""
    if utts_per_batch < 1:
        raise ValueError("utts_per_batch must be >= 1")
    utts = list(tokens.keys())
    out = []
    for s0 in range(0, len(utts), utts_per_batch):
        keys, rows, group, target, a, e = [], [], [], [], [], []
        for g, u in enumerate(utts[s0:s0 + utts_per_batch]):
            for h, toks in tokens[u].items():
                keys.append((u, h))
                rows.append([cls_id] + [int(t) for t in toks] + [sep_id])
                group.append(g)
                target.append(pll[u][h])
                a.append(am[u][h])
                e.append(cer[u][h])
        if not rows:
            continue
        T = max(len(r) for r in rows)
        ids = np.zeros((len(rows), T), np.int32)
        mask = np.zeros((len(rows), T), np.int32)
        for i, r in enumerate(rows):
            ids[i, :len(r)] = r
            mask[i, :len(r)] = 1
        out.append(dict(input_ids=ids, attention_mask=mask, group=np.asarray(group, np.int32),
                        target=np.asarray(target, np.float32), am=np.asarray(a, np.float32),
                        err=np.asarray(e, np.float32), keys=keys))
    return out


def batch_capacity(batches: List[dict]):
    """(max_rows, max_seq) a trainer needs for these batches."""
    return max(b["input_ids"].size for b in batches), max(b["input_ids"].shape[1] for b in batches)


def run_one_epoch(trainer: ClsTrainer, batches: List[dict], train_mode: bool, scores: Optional[Scores] = None) -> float:
    """One pass over the batches: forward + backward + AdamW step per batch (train_mode) or the loss only
    (eval: no dropout, no update).  Returns the mean of the batch losses; fills ``scores`` ({utt: {hyp:
    score}}) with the scores of each batch's forward pass when given."""
    total = 0.0
    for b in batches:
        loss, s = trainer.step(b["input_ids"], b["attention_mask"], b["group"], b["target"], b["am"], b["err"],
                               mode=1 if train_mode else 0)
        total += loss
        if scores is not None:
            for (u, h), v in zip(b["keys"], s.tolist()):
                scores.setdefault(u, {})[h] = v
    return total / max(len(batches), 1)


def train(state_dict, tokens, pll: Scores, am: Scores, cer: Scores, epochs: int = 1, lr: float = 1e-5,
          utts_per_batch: int = 4, md_weight: float = 1.0, mwer_weight: float = 0.0, am_weight: float = 1.0,
          dev: Optional[tuple] = None, cfg: Optional[dict] = None, device: int = 0, hidden_dropout: float = 0.1,
          attention_dropout: float = 0.1, seed: int = 0):
    """Train the student for ``epochs`` passes over (tokens, pll, am, cer); ``dev`` = the same four dicts
    of a held-out split, evaluated after every epoch.  One AdamW for the whole run.  Returns (the trained
    state_dict under the keys of ``state_dict``, {"train": [epoch losses], "dev": [...]})."""
    batches = make_batches(tokens, pll, am, cer, utts_per_batch)
    dev_batches = make_batches(*dev, utts_per_batch) if dev is not None else []
    max_rows, max_seq = batch_capacity(batches + dev_batches)
    losses = {"train": [], "dev": []}
    with ClsTrainer(state_dict, cfg, device=device, lr=lr, md_weight=md_weight, mwer_weight=mwer_weight,
                    am_weight=am_weight, hidden_dropout=hidden_dropout, attention_dropout=attention_dropout, seed=seed,
                    max_rows=max_rows, max_seq=max_seq) as tr:
        tr.reset_optimizer(lr)
        for _ in range(epochs):
            losses["train"].append(run_one_epoch(tr, batches, True))
            if dev_batches:
                losses["dev"].append(run_one_epoch(tr, dev_batches, False))
        return tr.state_dict(), losses
