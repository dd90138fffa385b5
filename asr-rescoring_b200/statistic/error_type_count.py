"""Edit-operation counts (the reference's ``statistic/error_type_count.py``).

The letters are the reference's (``espnet_data/preprocess/align.py``), and ``I`` / ``D`` are the
reverse of jiwer's naming (DESIGN.md §3.10):

====  ===========================================  ==================
op    meaning                                      textbook / jiwer
====  ===========================================  ==================
U     reference and hypothesis symbol are equal    hit
S     they differ                                  substitution
I     a reference symbol the hypothesis lacks      deletion
D     a hypothesis symbol the reference lacks      insertion
====  ===========================================  ==================

S + I + D of a pair is its character edit distance, so over a corpus
(S + I + D) / sum(len(ref)) is the CER of ``rescore.py``.

    python -m asr_rescoring_b200.statistic.error_type_count hyp_alignment.json
"""
from __future__ import annotations

import json
import sys
from typing import Dict, Sequence

import numpy as np

from .. import engine

OPS = ("U", "S", "I", "D")


def _as_dict(counts) -> Dict[str, int]:
    return {op: int(c) for op, c in zip(OPS, counts)}


def count_alignment(hyp_alignment: Dict[str, Dict[str, list]]) -> Dict[str, object]:
    """U/S/I/D totals over a hyp_alignment dict ({utt: {hyp_k: [aligned_ref, aligned_hyp, ops]}}):
    {"total": {op: n}, "per_rank": {hyp_k: {op: n}}}, ranks in order of first appearance."""
    total = dict.fromkeys(OPS, 0)
    per_rank: Dict[str, Dict[str, int]] = {}
    for hyps in hyp_alignment.values():
        for k, (_, _, ops) in hyps.items():
            rank = per_rank.setdefault(k, dict.fromkeys(OPS, 0))
            for op in ops:
                rank[op] += 1
                total[op] += 1
    return {"total": total, "per_rank": per_rank}


def error_counts(refs: Sequence[str], hyps: Sequence[str]) -> Dict[str, int]:
    """Corpus U/S/I/D of (refs[i], hyps[i]) pairs, aligned on the device in one launch (strings
    stripped as for the CER).  Fed the 1-best of ``rescore.get_highest_score_hyp`` at the best
    weight, it splits that CER into substitutions, missing (I) and extra (D) characters."""
    if len(refs) != len(hyps):
        raise ValueError("reference and hypothesis lists differ in length")
    if len(refs) == 0:
        return dict.fromkeys(OPS, 0)
    return _as_dict(engine.align(refs, hyps).counts.sum(axis=0, dtype=np.int64))


def main(argv=None) -> int:
    argv = sys.argv[1:] if argv is None else argv
    if len(argv) != 1:
        print("usage: error_type_count.py hyp_alignment.json", file=sys.stderr)
        return 2
    with open(argv[0], encoding="utf-8") as f:
        print(json.dumps(count_alignment(json.load(f)), indent=1))
    return 0


if __name__ == "__main__":
    sys.exit(main())
