"""Other reference call sites of ``jiwer.cer`` served by the warp-per-pair Levenshtein kernel
(SURVEY.md §8f rank 3):

* per-hypothesis CER of the upstream data prep — ``espnet_data/preprocess/main.py:59-60``
  (``hyps_cer.json``: {utt: {hyp_k: cer(ref, hyp_k)}});
* the CER utility of minimum-Bayes-risk decoding — ``RMBR/utility_functions.py:24-33``
  (``CerScoreFunction``: 1 - cer(ref, cand) for n*(n-1) pairs per utterance) and
  ``RMBR/mbr.py:5-27`` (``mbr_decode``).

Every pair of a call goes through ONE kernel launch; jiwer's per-pair semantics are kept:
strings stripped, characters = code points, CER = distance / len(reference), an empty
reference raises.
"""
from __future__ import annotations

from typing import Dict, List, Sequence

import numpy as np

from . import engine


def pair_cer(refs: Sequence[str], hyps: Sequence[str]) -> np.ndarray:
    """float64 [n]: jiwer.cer(refs[i], hyps[i]) for every i."""
    if len(refs) != len(hyps):
        raise ValueError("reference and hypothesis lists differ in length")
    lens = np.array([len(r.strip()) for r in refs], np.int64)
    if (lens == 0).any():
        raise ValueError("one or more references are empty strings")
    if len(refs) == 0:
        return np.zeros(0, np.float64)
    dist = engine.levenshtein(refs, hyps)
    return dist.astype(np.float64) / lens.astype(np.float64)


def hyps_cer(hyps_text: Dict[str, Dict[str, str]], ref_text: Dict[str, str]) -> Dict[str, Dict[str, float]]:
    """espnet_data/preprocess/main.py:51-60 for a whole split."""
    refs, hyps = [], []
    for utt, hs in hyps_text.items():
        for h in hs.values():
            refs.append(ref_text[utt])
            hyps.append(h)
    c = pair_cer(refs, hyps)
    out, i = {}, 0
    for utt, hs in hyps_text.items():
        out[utt] = {}
        for k in hs:
            out[utt][k] = float(c[i])
            i += 1
    return out


# The symbol an alignment puts opposite an unmatched one ('D' in aligned_ref, 'I' in aligned_hyp).
# The reference's own gap symbol is not recorded; the empty string cannot be a character of
# either side, and "".join(aligned_ref) gives back the (stripped) reference.
GAP = ""


def hyp_alignment(hyps_text: Dict[str, Dict[str, str]], ref_text: Dict[str, str]) -> Dict[str, Dict[str, list]]:
    """espnet_data/preprocess/main.py's hyp_alignment.json for a whole split, one kernel launch:
    {utt: {hyp_k: [aligned_ref, aligned_hyp, ops]}}, three lists of equal length per hypothesis
    over the characters of the stripped strings (DESIGN.md §3.10)."""
    utts = list(hyps_text)
    refs = [ref_text[u].strip() for u in utts]
    hyps, pair_ref = [], []
    for r, u in enumerate(utts):
        for h in hyps_text[u].values():
            hyps.append(h.strip())
            pair_ref.append(r)
    rc, ro = engine.pack_strings(refs)
    hc, ho = engine.pack_strings(hyps)
    pair_ref = np.asarray(pair_ref, np.int32)
    al = engine.align_packed(rc, ro, hc, ho, pair_ref)
    n = len(hyps)
    # the ops of every pair back to back, and the character each of them consumes on either side
    n_ops = al.n_ops.astype(np.int64)
    starts = np.zeros(n + 1, np.int64)
    np.cumsum(n_ops, out=starts[1:])
    pos = np.arange(int(starts[-1]), dtype=np.int64) - np.repeat(starts[:-1] - al.off[:-1], n_ops)
    ops = al.ops[pos]
    take_ref = ops != ord("D")
    take_hyp = ops != ord("I")
    na = np.diff(ro)[pair_ref]
    nb = np.diff(ho)
    base_ref = np.repeat(np.cumsum(na) - na, n_ops)        # ref characters consumed before each pair
    base_hyp = np.repeat(np.cumsum(nb) - nb, n_ops)
    i_ref = np.cumsum(take_ref) - take_ref - base_ref + np.repeat(ro[pair_ref], n_ops)
    i_hyp = np.cumsum(take_hyp) - take_hyp - base_hyp + np.repeat(ho[:-1], n_ops)
    ref_chars = np.array(list("".join(refs)) + [GAP], dtype=object)
    hyp_chars = np.array(list("".join(hyps)) + [GAP], dtype=object)
    a_ref = ref_chars[np.where(take_ref, i_ref, len(ref_chars) - 1)].tolist()
    a_hyp = hyp_chars[np.where(take_hyp, i_hyp, len(hyp_chars) - 1)].tolist()
    letters = list(ops.tobytes().decode("ascii"))
    out, p = {}, 0
    bounds = starts.tolist()
    for u in utts:
        out[u] = {}
        for k in hyps_text[u]:
            s, e = bounds[p], bounds[p + 1]
            out[u][k] = [a_ref[s:e], a_hyp[s:e], letters[s:e]]
            p += 1
    return out


class BaseFunction():
    def __init__(self, config) -> None:
        self.config = config

    def score(self):
        raise NotImplementedError


class CerScoreFunction(BaseFunction):
    """RMBR/utility_functions.py:24-33: similarity = 1 - cer(ref, cand)."""

    def score(self, cands, refs):
        return [1 - e for e in pair_cer(refs, cands).tolist()]


def mbr_decode(n_best: int, all_hyps: List[List[str]], utility_function: BaseFunction):
    """RMBR/mbr.py:5-27: expected-utility argmax over the top n_best hypotheses."""
    import torch
    cands, refs = [], []
    for utt_hyps in all_hyps:
        for hyp_i_pos in range(n_best):
            cands += [utt_hyps[hyp_i_pos]] * (n_best - 1)
            refs += utt_hyps[:hyp_i_pos] + utt_hyps[hyp_i_pos + 1:n_best]
    scores = utility_function.score(cands, refs)
    if not isinstance(scores, torch.Tensor):
        scores = torch.tensor(scores, dtype=torch.float)
    scores = scores.reshape(len(all_hyps), n_best, n_best - 1)
    scores = scores.sum(dim=-1)
    max_value_index = scores.argmax(dim=-1).cpu()
    predictions = [all_hyps[utt_id][v_index] for utt_id, v_index in enumerate(max_value_index)]
    return predictions, scores
