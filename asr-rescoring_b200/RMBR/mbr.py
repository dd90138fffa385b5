"""Minimum-Bayes-risk decoding over N-best lists from one within-utterance utility matrix.

``find_best_length`` is the dev sweep over the number k = 2 .. n_best of hypotheses that take part
in MBR (RMBR/main.py:15-35 of the reference, which is not in the reference tree): for each k,
hypothesis i < k of an utterance scores sum_{j < k, j != i} U[i, j] and the first argmax is chosen,
exactly what ``cer_clients.mbr_decode(k, hyps, utility)`` picks.  The pairwise matrix is computed
once (``BertScoreFunction.pairwise`` or any [N, n, n] array) and every k reads prefix sums of it;
the CERs come from one Levenshtein launch over all [N, n_best] candidates (rescore.pair_distances).

``expected_utility`` and ``utility_json`` turn the same matrix into {utt: {hyp: score}} that rescore.py
reads as its ``lm`` input with ``formula: "C"`` ((1-w)*am/len + w*lm, the combiner of the
reference's RMBR/BertScore runs).

There is no YAML front end: the reference's RMBR configuration files are not part of the reference
tree, so the functions take plain arguments.
"""
from __future__ import annotations

import json
import sys
from typing import Dict, Sequence, Tuple

import numpy as np


def expected_utility(U: np.ndarray, k: int | None = None) -> np.ndarray:
    """float64 [N, k]: sum over j < k, j != i of U[:, i, j] for every i < k (k defaults to n_best)."""
    U = np.asarray(U)
    n = U.shape[1] if k is None else int(k)
    V = U[:, :n, :n].astype(np.float64)
    return V.sum(axis=2) - np.diagonal(V, axis1=1, axis2=2)


def mbr_choices(U: np.ndarray) -> Dict[int, np.ndarray]:
    """{k: int64 [N] first argmax of the expected utility over the first k hypotheses} for k = 2 .. n_best,
    from prefix sums over j of one [N, n_best, n_best] matrix."""
    U = np.asarray(U, np.float64)
    n = U.shape[1]
    V = U * (1.0 - np.eye(n))[None]          # a hypothesis is not its own reference
    prefix = np.cumsum(V, axis=2)            # prefix[u, i, k-1] = sum_{j < k} V[u, i, j]
    return {k: np.argmax(prefix[:, :k, k - 1], axis=1) for k in range(2, n + 1)}


def find_best_length(all_hyps: Sequence[Sequence[str]], refs: Sequence[str], n_best: int, utility,
                     U: np.ndarray | None = None) -> Tuple[int, Dict[int, float]]:
    """(best k, {k: corpus CER of the MBR choice with k hypotheses}) on a dev split; the first k with
    the strictly smallest CER wins, as rescore.find_best_weight does for the weight.  ``utility`` needs
    ``pairwise(all_hyps, n_best)`` unless the matrix ``U`` is given."""
    from .. import rescore
    if U is None:
        U = utility.pairwise(all_hyps, n_best)
    total = 0
    for r in refs:
        if len(r.strip()) == 0:
            raise ValueError("one or more references are empty strings")
        total += len(r.strip())
    dist = rescore.pair_distances([list(h[:n_best]) for h in all_hyps], list(refs), n_best)
    rows = np.arange(len(refs))
    cers, best_k, best_cer = {}, None, sys.float_info.max
    for k, arg in mbr_choices(U).items():
        cer = float(int(dist[rows, arg].sum())) / float(total)
        cers[k] = cer
        if cer < best_cer:
            best_k, best_cer = k, cer
    return best_k, cers


def utility_json(utt_ids: Sequence[str], E: np.ndarray, hyp_ids: Sequence[Sequence[str]] | None = None
                 ) -> Dict[str, Dict[str, float]]:
    """{utt: {hyp_k: expected utility}} from [N, n] scores (hyp ids default to hyp_1 .. hyp_n)."""
    E = np.asarray(E, np.float64)
    out = {}
    for u, utt in enumerate(utt_ids):
        ids = hyp_ids[u] if hyp_ids is not None else [f"hyp_{k + 1}" for k in range(E.shape[1])]
        out[utt] = {h: float(E[u, k]) for k, h in enumerate(ids)}
    return out


def write_utility_json(path: str, utt_ids: Sequence[str], E: np.ndarray,
                       hyp_ids: Sequence[Sequence[str]] | None = None) -> None:
    """utility_json written as rescore.py's dev_lm_path / test_lm_path input."""
    with open(path, "w", encoding="utf-8") as f:
        json.dump(utility_json(utt_ids, E, hyp_ids), f, ensure_ascii=False, indent=1)
