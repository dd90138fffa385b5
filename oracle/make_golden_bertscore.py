"""Generate tests/golden/bertscore_golden.json with the fp32 restatement of bert_score's recall.

    python oracle/make_golden_bertscore.py        (CPU only; a few seconds)

oracle/bertscore_oracle.py is the pin (bert_score is not installed; RMBR/ is not in the reference
tree).  Two cases, each the within-utterance recall matrix U[u, i, j] = R(h_i, h_j) of every ordered
pair i != j (diagonal 0), hypotheses tokenised with tokenizer.SyntheticCharTokenizer:

  * tiny: BERT_TINY, perturbed random init (seed 10), both layers; 3 utterances x 5 hypotheses with
    an empty hypothesis, duplicate strings (within and across utterances) and a 1-token hypothesis;
  * base: bert-base-chinese shape, default random init (seed 10), 8 layers; 20 synthetic AISHELL-shaped
    utterances x 10-best (synth.make_nbest, seed 7).
"""
from __future__ import annotations

import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import bertscore_oracle  # noqa: E402
from asr_rescoring_b200 import synth  # noqa: E402
from asr_rescoring_b200.tokenizer import SyntheticCharTokenizer  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "bertscore_golden.json")


def tiny_hyps():
    nb = synth.make_nbest(3, 5, seed=5)
    hyps = [list(h) for h in nb.hyps]
    hyps[0][3] = ""                    # empty hypothesis
    hyps[0][4] = hyps[0][1]            # duplicate within an utterance
    hyps[1][2] = hyps[1][2][:1]        # one token
    hyps[2][4] = " " + hyps[0][0]      # duplicate across utterances (equal after strip())
    return hyps


def pairwise(sd, cfg, hyps, num_layers):
    tok = SyntheticCharTokenizer()
    util = bertscore_oracle.OracleBertScore(sd, cfg, lambda s: tok.encode(s), num_layers)
    n = len(hyps[0])
    cands, refs = [], []
    for hs in hyps:
        for i in range(n):
            for j in range(n):
                if i != j:
                    cands.append(hs[i])
                    refs.append(hs[j])
    U = np.zeros((len(hyps), n, n))
    U[:, ~np.eye(n, dtype=bool)] = np.asarray(util.score(cands, refs)).reshape(len(hyps), n * (n - 1))
    return U


def main():
    cases = []
    specs = [("tiny", synth.BERT_TINY, 10, True, 2, tiny_hyps()),
             ("base", synth.BERT_BASE_CHINESE, 10, False, 8, synth.make_nbest(20, 10, seed=7).hyps)]
    for name, cfg, seed, perturb, nl, hyps in specs:
        sd = synth.random_init_state_dict(cfg, seed, perturb)
        U = pairwise(sd, cfg, hyps, nl)
        cases.append(dict(name=name, cfg=cfg, seed=seed, perturb=perturb, num_layers=nl, hyps=hyps,
                          recall=U.round(7).tolist()))
        print(f"{name}: {U.size} entries, recall range [{U.min():.4f}, {U.max():.4f}]")
    with open(GOLD, "w", encoding="utf-8") as f:
        json.dump(dict(generator="oracle/make_golden_bertscore.py", cases=cases), f, ensure_ascii=False)
        f.write("\n")


if __name__ == "__main__":
    main()
