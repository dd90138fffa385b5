"""Drop-in for the scoring use of the reference's ``RescoreBert/model.py`` (SURVEY.md §8f rank 2).

``RescoreBert(state_dict)`` stands in for ``RescoreBert(bert)`` + ``load_state_dict(checkpoint)`` +
``.to(device)`` (RescoreBert/main.py:249-252): the checkpoint is the state_dict of the
reference's module — ``bert.*`` (a transformers BertModel) plus ``linear.weight`` [1, H] and
``linear.bias`` [1] (RescoreBert/model.py:7-11).  ``score_packed`` / ``__call__`` replace the
forward (model.py:13-21) and the padded batches of RescoreBert/main.py:31-75: every hypothesis
runs once through the B200 encoder as ``[CLS] t [SEP]`` (varlen packed, no padding) and
``lm_score = Linear([CLS] state)``.  Training the student on the teacher's PLLs (MD and MWER losses;
MWED is not built) is ``RescoreBert/train.py``; the state_dict it returns loads here directly.
"""
from __future__ import annotations

from typing import Dict, Sequence

import numpy as np

from ..engine import PllScorer


class RescoreBert:
    def __init__(self, state_dict, cfg=None, device: int = 0, max_chunk_tokens: int = 0, operand_dtype: str = "bf16"):
        self.linear_w = state_dict["linear.weight"].detach().float().cpu().numpy().reshape(-1)
        self.linear_b = float(state_dict["linear.bias"].detach().float().cpu().reshape(-1)[0])
        enc = {k: v for k, v in state_dict.items() if k.startswith("bert.") and not k.startswith("bert.pooler")}
        self.encoder = PllScorer(enc, cfg, device=device, max_chunk_tokens=max_chunk_tokens, operand_dtype=operand_dtype)

    def score_packed(self, tokens: np.ndarray, offsets: np.ndarray) -> np.ndarray:
        """tokens: wordpiece ids without specials, packed; offsets int64[n+1] -> float32[n]."""
        return self.encoder.score_cls_packed(tokens, offsets, self.linear_w, self.linear_b)

    def score_hyps(self, hyps: Dict[str, Dict[str, Sequence[int]]]) -> Dict[str, Dict[str, float]]:
        """{utt: {hyp: token ids}} -> {utt: {hyp: lm_score}} (the dev_lm.json / test_lm.json content
        of RescoreBert/main.py:254-283)."""
        flat, off = [], [0]
        for hs in hyps.values():
            for toks in hs.values():
                flat.extend(toks)
                off.append(len(flat))
        sc = self.score_packed(np.asarray(flat, np.int32), np.asarray(off, np.int64))
        out, i = {}, 0
        for u, hs in hyps.items():
            out[u] = {}
            for h in hs:
                out[u][h] = float(sc[i])
                i += 1
        return out

    def close(self):
        self.encoder.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()
