"""BERTScore-recall utility of RMBR (RMBR/utility_functions.py:9-23 of the reference) on the device.

The reference calls ``bert_score.score(cands, refs, lang="zh")`` with default arguments; neither
RMBR/ nor ``bert_score`` is in the reference tree or installed, so the definition implemented here
is this project's contract (include/pllb.h, pllb_embed / pllb_bertscore; DESIGN.md §3.9):

    R(c, r) = mean over the wordpieces x of r of max over all positions y of [CLS] c [SEP]
              of cos(E_r[x], E_c[y]),  E = fp32 output of encoder layer ``num_layers``,
    R = 0 when either string is empty after strip().

``score(cands, refs)`` keeps the reference signature, so ``cer_clients.mbr_decode(n, hyps,
BertScoreFunction(...))`` works unchanged:

    from asr_rescoring_b200.RMBR.utility_functions import BertScoreFunction
    from asr_rescoring_b200.cer_clients import mbr_decode
    util = BertScoreFunction(bert_state_dict, tokenizer, num_layers=8)
    best, expected = mbr_decode(10, all_hyps, util)
"""
from __future__ import annotations

from typing import Dict, List, Sequence, Tuple

import numpy as np

from .. import engine
from ..cer_clients import BaseFunction

DEFAULT_MAX_ROWS = 1 << 20      # embedding rows per block: 3 GiB of fp32 states at hidden 768


def dedup_pairs(cands: Sequence[str], refs: Sequence[str]) -> Tuple[List[str], np.ndarray, np.ndarray]:
    """Stripped unique strings in order of first appearance (candidates and references interleaved
    pair by pair) and the int32 index of every pair's candidate and reference into them."""
    if len(cands) != len(refs):
        raise ValueError("candidate and reference lists differ in length")
    index: Dict[str, int] = {}
    cand = np.empty(len(cands), np.int32)
    ref = np.empty(len(refs), np.int32)
    for p, (c, r) in enumerate(zip(cands, refs)):
        cand[p] = index.setdefault(c.strip(), len(index))
        ref[p] = index.setdefault(r.strip(), len(index))
    return list(index), cand, ref


def plan_blocks(cand: np.ndarray, ref: np.ndarray, seq_rows: np.ndarray, max_rows: int):
    """Split the pairs into consecutive blocks whose sequences need at most ``max_rows`` embedding rows
    (a block always takes at least one pair).  Yields (pair slice, global sequence ids of the block in
    order of first use, local cand, local ref)."""
    n = len(cand)
    p = 0
    while p < n:
        local: Dict[int, int] = {}
        rows = 0
        q = p
        while q < n:
            new = [s for s in dict.fromkeys((int(cand[q]), int(ref[q]))) if s not in local]
            add = int(sum(seq_rows[s] for s in new))
            if q > p and rows + add > max_rows:
                break
            for s in new:
                local[s] = len(local)
            rows += add
            q += 1
        lc = np.fromiter((local[int(s)] for s in cand[p:q]), np.int32, q - p)
        lr = np.fromiter((local[int(s)] for s in ref[p:q]), np.int32, q - p)
        yield slice(p, q), np.fromiter(local, np.int64, len(local)), lc, lr
        p = q


class BertScoreFunction(BaseFunction):
    """``score(cands, refs)`` -> BERTScore recall of every pair; ``pairwise`` -> the within-utterance
    recall matrices.  ``state_dict``: the ``bert.*`` tensors PllScorer takes (pooler and MLM head are
    not needed); ``tokenizer``: a tokenizer.py tokenizer (``encode_batch`` is used);
    ``max_rows`` bounds the embedding rows held at once (pairs go in consecutive blocks)."""

    def __init__(self, state_dict, tokenizer, num_layers: int = 8, cfg=None, device: int = 0,
                 operand_dtype: str = "bf16", max_rows: int = DEFAULT_MAX_ROWS, max_chunk_tokens: int = 0):
        super().__init__(dict(num_layers=num_layers, operand_dtype=operand_dtype, max_rows=max_rows))
        self.scorer = engine.PllScorer(state_dict, cfg, device=device, max_chunk_tokens=max_chunk_tokens,
                                       operand_dtype=operand_dtype)
        if not 0 <= num_layers <= self.scorer.cfg["num_layers"]:
            raise ValueError(f"num_layers must be in [0, {self.scorer.cfg['num_layers']}]")
        self.tokenizer = tokenizer
        self.num_layers = int(num_layers)
        self.max_rows = int(max_rows)
        self.device = device

    def close(self):
        self.scorer.close()

    def score(self, cands: Sequence[str], refs: Sequence[str]) -> List[float]:
        """R(cands[p], refs[p]) for every p (bert_score.score(...)[1] of the reference's call)."""
        from ..tokenizer import encode_batch
        uniq, cand, ref = dedup_pairs(cands, refs)
        if len(cand) == 0:
            return []
        ids, off = encode_batch(self.tokenizer, uniq)
        return self._recall(ids, off, cand, ref).tolist()

    def _recall(self, ids: np.ndarray, off: np.ndarray, cand: np.ndarray, ref: np.ndarray) -> np.ndarray:
        """float32 recall of the pairs (cand, ref) over the token lists (ids, off)."""
        import torch
        dev = torch.device("cuda", self.device)
        out = np.empty(len(cand), np.float32)
        seq_rows = np.diff(off) + 2
        for sl, seqs, lc, lr in plan_blocks(cand, ref, seq_rows, self.max_rows):
            lens = np.diff(off)[seqs]
            b_off = np.zeros(len(seqs) + 1, np.int64)
            np.cumsum(lens, out=b_off[1:])
            tok = np.concatenate([ids[off[s]:off[s + 1]] for s in seqs]).astype(np.int32) if b_off[-1] else \
                np.zeros(1, np.int32)
            t = torch.from_numpy(tok).to(dev)
            emb = self.scorer.embed(t, b_off, self.num_layers)
            row_off = b_off + 2 * np.arange(len(seqs) + 1, dtype=np.int64)
            out[sl] = self.scorer.bertscore(emb, row_off, lc, lr).cpu().numpy()
            del emb, t
        return out

    def pairwise(self, all_hyps: Sequence[Sequence[str]], n_best: int) -> np.ndarray:
        """float32 [N, n_best, n_best]: U[u, i, j] = R(h_i, h_j) of utterance u for i != j; the diagonal
        is 0 (a hypothesis is not scored against itself, as in mbr_decode)."""
        n = int(n_best)
        cands, refs = [], []
        for hs in all_hyps:
            if len(hs) < n:
                raise ValueError("every utterance needs at least n_best hypotheses")
            for i in range(n):
                for j in range(n):
                    if j != i:
                        cands.append(hs[i])
                        refs.append(hs[j])
        U = np.zeros((len(all_hyps), n, n), np.float32)
        if n > 1 and len(all_hyps):
            off_diag = ~np.eye(n, dtype=bool)
            U[:, off_diag] = np.asarray(self.score(cands, refs), np.float32).reshape(len(all_hyps), n * (n - 1))
        return U
