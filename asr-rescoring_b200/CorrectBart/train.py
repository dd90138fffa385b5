"""CorrectBart fine-tuning on (1-best hypothesis, reference) pairs.

The encoder reads ``[CLS] hyp [SEP]``, the labels are ``[CLS] ref [SEP]``; the step is
``BartForConditionalGeneration.forward(labels=...)`` + ``loss.backward()`` + ``torch.optim.AdamW``, run by
``engine.Seq2SeqTrainer`` (include/pllb.h, ``pllb_s2s_train_*``, states the contract):

    from asr_rescoring_b200.CorrectBart.train import one_hyp_pairs, train
    from asr_rescoring_b200.CorrectBart.model import CorrectBart, compute_cer
    hyps, refs = one_hyp_pairs(hyps_text, ref_text)
    sd, losses = train(state_dict, cfg, tokenizer, hyps, refs, epochs=3, lr=1e-5, sents_per_batch=32)
    model = CorrectBart(sd, cfg, tokenizer)
    print(compute_cer(model.correct(dev_hyps), dev_refs))

There is no YAML front end: the reference's training configuration is not part of the reference tree, so the
driver takes plain arguments.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from ..engine import Seq2SeqTrainer


def one_hyp_pairs(hyps_text: Dict[str, Dict[str, str]], ref_text: Dict[str, str]) -> Tuple[List[str], List[str]]:
    """(1-best hypotheses, references) in utterance order: hyp_1 of every utterance of ``hyps_text`` with the
    reference of the same utterance."""
    missing = [u for u in hyps_text if u not in ref_text]
    if missing:
        raise ValueError(f"{len(missing)} utterances have no reference, e.g. {missing[0]!r}")
    utts = list(hyps_text)
    return [hyps_text[u]["hyp_1"] for u in utts], [ref_text[u] for u in utts]


def make_batches(tokenizer, hyps: Sequence[str], refs: Sequence[str], sents_per_batch: int, label_pad: int = -100,
                 cls_id: int = 101, sep_id: int = 102, pad_id: int = 0) -> List[dict]:
    """Batches of ``sents_per_batch`` pairs in input order: input_ids / attention_mask int32 [B, T_enc]
    (``[CLS] hyp [SEP]``, right-padded with pad_id) and labels int32 [B, T_dec] (``[CLS] ref [SEP]``, padded
    with ``label_pad``).  The default -100 leaves the padding out of the loss; ``label_pad=pad_id`` counts it, as
    transformers then does."""
    if sents_per_batch < 1:
        raise ValueError("sents_per_batch must be >= 1")
    if len(hyps) != len(refs):
        raise ValueError("hypothesis and reference lists differ in length")
    out = []
    for s0 in range(0, len(hyps), sents_per_batch):
        enc = [[cls_id] + list(tokenizer.encode(h)) + [sep_id] for h in hyps[s0:s0 + sents_per_batch]]
        dec = [[cls_id] + list(tokenizer.encode(r)) + [sep_id] for r in refs[s0:s0 + sents_per_batch]]
        Te, Td = max(map(len, enc)), max(map(len, dec))
        ids = np.full((len(enc), Te), pad_id, np.int32)
        mask = np.zeros((len(enc), Te), np.int32)
        labels = np.full((len(dec), Td), label_pad, np.int32)
        for i, (e, d) in enumerate(zip(enc, dec)):
            ids[i, :len(e)] = e
            mask[i, :len(e)] = 1
            labels[i, :len(d)] = d
        out.append(dict(input_ids=ids, attention_mask=mask, labels=labels))
    return out


def batch_capacity(batches: List[dict]) -> Tuple[int, int, int]:
    """(max_batch, max_enc_len, max_dec_len) a trainer needs for these batches."""
    return (max(b["input_ids"].shape[0] for b in batches), max(b["input_ids"].shape[1] for b in batches),
            max(b["labels"].shape[1] for b in batches))


def run_one_epoch(trainer: Seq2SeqTrainer, batches: List[dict], train_mode: bool) -> float:
    """One pass: forward + backward + AdamW step per batch (train_mode) or the loss only (eval: no dropout, no
    update).  Returns the mean of the batch losses."""
    total = 0.0
    for b in batches:
        total += trainer.step(b["input_ids"], b["attention_mask"], b["labels"], mode=1 if train_mode else 0)
    return total / max(len(batches), 1)


def train(state_dict, cfg: dict, tokenizer, hyps: Sequence[str], refs: Sequence[str], epochs: int = 1, lr: float = 1e-5,
          sents_per_batch: int = 32, dev: Optional[Tuple[Sequence[str], Sequence[str]]] = None, device: int = 0,
          dropout: Optional[float] = None, attention_dropout: Optional[float] = None, seed: int = 0,
          weight_decay: float = 0.01, label_pad: int = -100):
    """Fine-tune for ``epochs`` passes over (hyps, refs); ``dev`` = (hyps, refs) of a held-out split, evaluated
    after every epoch.  One AdamW for the whole run.  Returns (the trained state_dict under the keys of
    ``state_dict``, {"train": [epoch losses], "dev": [...]}); ``CorrectBart(sd, cfg, tokenizer)`` decodes with it."""
    pad_id = int(cfg.get("pad_token_id") or 0)
    batches = make_batches(tokenizer, hyps, refs, sents_per_batch, label_pad, pad_id=pad_id)
    dev_batches = make_batches(tokenizer, *dev, sents_per_batch, label_pad, pad_id=pad_id) if dev is not None else []
    max_batch, max_enc, max_dec = batch_capacity(batches + dev_batches)
    losses = {"train": [], "dev": []}
    with Seq2SeqTrainer(state_dict, cfg, device=device, lr=lr, dropout=dropout, attention_dropout=attention_dropout,
                        seed=seed, max_batch=max_batch, max_enc_len=max_enc, max_dec_len=max_dec,
                        weight_decay=weight_decay) as tr:
        for _ in range(epochs):
            losses["train"].append(run_one_epoch(tr, batches, True))
            if dev_batches:
                losses["dev"].append(run_one_epoch(tr, dev_batches, False))
        return tr.state_dict(), losses
