"""CPU restatement (plain torch fp32) of RMBR's BERTScore-recall utility and its MBR decoding.

TEST INFRASTRUCTURE ONLY — imported by tests/ and tools/; never by the product path.

Provenance.  RMBR/utility_functions.py:9-23 calls bert_score.score(cands, refs, lang="zh") with its
default arguments, but neither RMBR/ nor the third-party bert_score package is in the reference tree or
installed.  What follows restates bert_score's scoring for those arguments and is the contract of
pllb_embed / pllb_bertscore (include/pllb.h), pinned by this restatement and not by a reference golden:

  * model ........ transformers.BertModel carrying the given state_dict, encoder truncated to num_layers
                   layers (bert_score: model.encoder.layer = layer[:num_layers]; 8 for bert-base-chinese
                   in its model table); embeddings = model(...)[0], fp32, every position of [CLS] t [SEP]
  * idf .......... idf=False: uniform weight 1, except [CLS] and [SEP] which get 0 (idf_dict)
  * matching ..... greedy_cos_idf: L2-normalise rows, similarity = hyp @ ref^T, multiplied by the padding
                   mask; recall = sum over ref rows of idf * max over hyp rows, divided by sum idf
  * empty ........ a sentence with only [CLS] [SEP] gives P = R = 0 (hyp_zero_mask / ref_zero_mask)
  * MBR .......... RMBR/mbr.py:5-27 (mbr_decode) and the k = 2 .. n_best sweep of RMBR/main.py:15-35

The contract scores each pair on its own (``recall_pairs``), so the maximum runs over real positions
only; ``greedy_cos_idf`` keeps bert_score's padded form, which returns 0 instead of a negative maximum.
"""
from __future__ import annotations

from typing import List, Sequence

import numpy as np
import torch


def bert_model(sd, cfg, num_layers: int):
    """fp32 transformers.BertModel with the ``bert.*`` tensors of sd, encoder truncated to num_layers."""
    from transformers import BertConfig, BertModel
    conf = BertConfig(vocab_size=cfg["vocab"], hidden_size=cfg["hidden"], num_hidden_layers=cfg["num_layers"],
                      num_attention_heads=cfg["num_heads"], intermediate_size=cfg["intermediate"],
                      max_position_embeddings=cfg["max_position"], type_vocab_size=cfg.get("type_vocab", 2),
                      layer_norm_eps=cfg.get("ln_eps", 1e-12), pad_token_id=0, hidden_act="gelu",
                      hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0)
    conf._attn_implementation = "eager"
    m = BertModel(conf, add_pooling_layer=False)
    enc = {k[len("bert."):]: v for k, v in sd.items() if k.startswith("bert.") and not k.startswith("bert.pooler.")}
    missing, unexpected = m.load_state_dict(enc, strict=False)
    assert not unexpected and all("position_ids" in k for k in missing), (missing, unexpected)
    m.encoder.layer = m.encoder.layer[:num_layers]
    return m.eval()


@torch.no_grad()
def embed(model, token_lists: Sequence[Sequence[int]], cls_id=101, sep_id=102, batch_size: int = 64) -> List[torch.Tensor]:
    """[L+2, H] fp32 states of every [CLS] t [SEP] (zero-padded batches with an attention mask)."""
    out = []
    for s0 in range(0, len(token_lists), batch_size):
        rows = [[cls_id] + list(t) + [sep_id] for t in token_lists[s0:s0 + batch_size]]
        T = max(len(r) for r in rows)
        ids = torch.zeros(len(rows), T, dtype=torch.long)
        am = torch.zeros(len(rows), T, dtype=torch.long)
        for i, r in enumerate(rows):
            ids[i, :len(r)] = torch.tensor(r)
            am[i, :len(r)] = 1
        hid = model(input_ids=ids, attention_mask=am)[0]
        out += [hid[i, :len(r)].clone() for i, r in enumerate(rows)]
    return out


def greedy_cos_idf(ref_embedding, ref_masks, ref_idf, hyp_embedding, hyp_masks, hyp_idf):
    """bert_score.utils.greedy_cos_idf (padded batch [B, T, H], masks / idf [B, T]) -> (P, R, F)."""
    ref_embedding = ref_embedding / torch.norm(ref_embedding, dim=-1).unsqueeze(-1)
    hyp_embedding = hyp_embedding / torch.norm(hyp_embedding, dim=-1).unsqueeze(-1)
    sim = torch.bmm(hyp_embedding, ref_embedding.transpose(1, 2))
    masks = torch.bmm(hyp_masks.unsqueeze(2).float(), ref_masks.unsqueeze(1).float())
    sim = sim * masks
    word_precision = sim.max(dim=2)[0]
    word_recall = sim.max(dim=1)[0]
    hyp_idf = hyp_idf / hyp_idf.sum(dim=1, keepdim=True)
    ref_idf = ref_idf / ref_idf.sum(dim=1, keepdim=True)
    P = (word_precision * hyp_idf).sum(dim=1)
    R = (word_recall * ref_idf).sum(dim=1)
    F = 2 * P * R / (P + R)
    hyp_zero = hyp_masks.sum(dim=1).eq(2)
    ref_zero = ref_masks.sum(dim=1).eq(2)
    P, R = P.masked_fill(hyp_zero, 0.0), R.masked_fill(hyp_zero, 0.0)
    P, R = P.masked_fill(ref_zero, 0.0), R.masked_fill(ref_zero, 0.0)
    F = F.masked_fill(torch.isnan(F) | hyp_zero | ref_zero, 0.0)
    return P, R, F


def pad_batch(embs: Sequence[torch.Tensor]):
    """Padded [B, T, H] states, masks and bert_score's uniform idf ([CLS] / [SEP] weight 0).  The padded
    rows hold ones: in bert_score they are the model's outputs at [PAD] positions, never zero vectors."""
    T = max(e.shape[0] for e in embs)
    H = embs[0].shape[1]
    E = torch.ones(len(embs), T, H)
    mask = torch.zeros(len(embs), T)
    idf = torch.zeros(len(embs), T)
    for i, e in enumerate(embs):
        E[i, :e.shape[0]] = e
        mask[i, :e.shape[0]] = 1
        idf[i, 1:e.shape[0] - 1] = 1
    return E, mask, idf


def recall_pairs(embs: Sequence[torch.Tensor], cand: Sequence[int], ref: Sequence[int]) -> np.ndarray:
    """float64 [n_pairs] R(embs[cand[p]], embs[ref[p]]), each pair in a batch of its own (no padding)."""
    out = np.zeros(len(cand), np.float64)
    for p, (c, r) in enumerate(zip(cand, ref)):
        Er, mr, ir = pad_batch([embs[r]])
        Ec, mc, ic = pad_batch([embs[c]])
        out[p] = float(greedy_cos_idf(Er, mr, ir, Ec, mc, ic)[1][0])
    return out


class OracleBertScore:
    """Utility with the reference's ``score(cands, refs)`` signature over token lists from ``encode``."""

    def __init__(self, sd, cfg, encode, num_layers: int):
        self.model = bert_model(sd, cfg, num_layers)
        self.encode = encode

    def score(self, cands, refs) -> List[float]:
        uniq = list(dict.fromkeys([s.strip() for s in list(cands) + list(refs)]))
        index = {s: i for i, s in enumerate(uniq)}
        embs = embed(self.model, [self.encode(s) for s in uniq])
        return recall_pairs(embs, [index[c.strip()] for c in cands], [index[r.strip()] for r in refs]).tolist()


def mbr_decode(n_best: int, all_hyps, utility):
    """RMBR/mbr.py:5-27: (predictions, expected utilities [N, n_best] as torch fp32)."""
    cands, refs = [], []
    for utt_hyps in all_hyps:
        for i in range(n_best):
            cands += [utt_hyps[i]] * (n_best - 1)
            refs += utt_hyps[:i] + utt_hyps[i + 1:n_best]
    scores = torch.tensor(utility.score(cands, refs), dtype=torch.float).reshape(len(all_hyps), n_best, n_best - 1)
    scores = scores.sum(dim=-1)
    idx = scores.argmax(dim=-1)
    return [all_hyps[u][int(i)] for u, i in enumerate(idx)], scores


def find_best_length(all_hyps, refs, n_best: int, utility):
    """RMBR/main.py:15-35: mbr_decode once per k = 2 .. n_best, corpus CER of each, first strict minimum."""
    from oracle import levenshtein_strings
    total = sum(len(r.strip()) for r in refs)
    cers, best_k, best = {}, None, float("inf")
    for k in range(2, n_best + 1):
        pred, _ = mbr_decode(k, all_hyps, utility)
        cer = float(int(levenshtein_strings([r.strip() for r in refs], [p.strip() for p in pred]).sum())) / total
        cers[k] = cer
        if cer < best:
            best_k, best = k, cer
    return best_k, cers
