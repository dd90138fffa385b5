"""Deterministic synthetic AISHELL-1-shaped N-best lists and random-init weights.

The reference ships no hypothesis text and no checkpoints (SURVEY.md §2 row 12,
§4), and nothing under /root/reference exists on the GPU box, so benchmarks and
parity tests use data synthesised from statistics of the reference's fixtures
(recorded below as plain numbers) following SURVEY.md §8(d):

  * utterance lengths: the length list of espnet_data/alfred/test/ref_text.json in
    utterance order (7 176 refs, 104 765 chars, min 3 / mean 14.6 / max 37) —
    data/aishell1_test_shape.json, written by tools/make_synth_shape.py;
  * per-hypothesis edit counts: round(hyps_cer * len(ref)) of
    espnet_data/alfred/test/hyps_cer.json per (utterance, k) from the same table
    (71 760 entries); hypotheses 11..50 and the length-stretched config 4 draw
    from its histogram;
  * AM scores: first-best mean/std and mean successive gaps of
    espnet_data/alfred/test/hyps_score.json;
  * token ids: no vocab.txt offline -> id = 670 + rank(char) mod 7322, inside
    the CJK block of bert-base-chinese; specials as in that vocab;
  * weights: BertForMaskedLM default init (N(0, 0.02), LayerNorm 1/0, zero
    biases, zero [PAD] row) under a fixed seed, keyed like the HF state_dict
    that MLM_PLL/main.py:185-186 loads.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List

import numpy as np

# espnet_data/alfred/test/ref_text.json: {len: count}
REF_LEN_HIST = {3: 1, 4: 2, 5: 7, 6: 61, 7: 81, 8: 121, 9: 531, 10: 669, 11: 581, 12: 615,
                13: 597, 14: 521, 15: 536, 16: 447, 17: 450, 18: 392, 19: 387, 20: 357,
                21: 329, 22: 233, 23: 150, 24: 85, 25: 15, 26: 3, 27: 3, 36: 1, 37: 1}
# espnet_data/alfred/test/hyps_cer.json: {edit distance: count}
EDIT_HIST = {0: 5276, 1: 37666, 2: 15901, 3: 6977, 4: 3250, 5: 1439, 6: 764, 7: 293,
             8: 120, 9: 53, 10: 9, 11: 11, 12: 1}
# espnet_data/alfred/test/hyps_score.json
AM_FIRST_MEAN, AM_FIRST_STD, AM_FIRST_MAX = -2.40, 2.08, -0.23
AM_GAP_MEAN = [2.04, 0.81, 0.46, 0.36, 0.26, 0.23, 0.19, 0.18, 0.23]
N_DISTINCT_CHARS = 2633

PAD_ID, UNK_ID, CLS_ID, SEP_ID, MASK_ID = 0, 100, 101, 102, 103

BERT_BASE_CHINESE = dict(num_layers=12, hidden=768, num_heads=12, intermediate=3072,
                         vocab=21128, max_position=512, type_vocab=2, ln_eps=1e-12)
BERT_LARGE_SHAPED = dict(num_layers=24, hidden=1024, num_heads=16, intermediate=4096,
                         vocab=21128, max_position=512, type_vocab=2, ln_eps=1e-12)
# smallest shape the kernels accept (hidden % 256 == 0, head dim 64); vocab is
# deliberately not a multiple of the vocab tile.
BERT_TINY = dict(num_layers=2, hidden=256, num_heads=4, intermediate=1024,
                 vocab=8000, max_position=128, type_vocab=2, ln_eps=1e-12)


def char_of_rank(rank: int) -> str:
    return chr(0x4E00 + (rank * 7) % 20000)


def synthetic_token_id(ch: str) -> int:
    """Deterministic char -> wordpiece id stand-in (SURVEY.md §8d)."""
    rank = ((ord(ch) - 0x4E00) * 17143) % 20000 if 0x4E00 <= ord(ch) < 0x4E00 + 20000 else ord(ch)
    return 670 + rank % 7322


@dataclass
class SynthNbest:
    utt_ids: List[str]
    refs: List[str]
    hyps: List[List[str]]              # [N][n_best]
    am: np.ndarray                     # float64 [N, n_best], descending per row
    edits: np.ndarray                  # int32 [N, n_best] number of random edits applied
    meta: dict = field(default_factory=dict)

    @property
    def n_best(self) -> int:
        return self.am.shape[1]

    def hyps_text(self) -> Dict[str, Dict[str, str]]:
        return {u: {f"hyp_{k + 1}": h for k, h in enumerate(hs)} for u, hs in zip(self.utt_ids, self.hyps)}

    def hyps_score(self) -> Dict[str, Dict[str, float]]:
        return {u: {f"hyp_{k + 1}": float(a) for k, a in enumerate(row)} for u, row in zip(self.utt_ids, self.am)}

    def ref_text(self) -> Dict[str, str]:
        return dict(zip(self.utt_ids, self.refs))

    def packed_tokens(self, vocab: int | None = None):
        """(int32 tokens, int64 offsets) over hyps in (utt, k) order."""
        flat = [h for hs in self.hyps for h in hs]
        off = np.zeros(len(flat) + 1, np.int64)
        np.cumsum([len(h) for h in flat], out=off[1:])
        tok = np.fromiter((synthetic_token_id(c) for h in flat for c in h), np.int32, int(off[-1]))
        if vocab is not None and vocab < 670 + 7322:
            tok = (104 + (tok % (vocab - 104))).astype(np.int32)
        return tok, off


_SHAPE = None


def shape_table():
    """(ref_len int64[7176], edits int64[7176, 10]) of the AISHELL-1 test set, utterance order."""
    global _SHAPE
    if _SHAPE is None:
        import json
        import os
        p = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "aishell1_test_shape.json")
        d = json.load(open(p))
        ref_len = np.array(d["ref_len"], np.int64)
        edits = np.array([[int(c, 36) for c in row] for row in d["edits_base36_per_utt"]], np.int64)
        assert ref_len.shape == (7176,) and edits.shape == (7176, 10)
        _SHAPE = (ref_len, edits)
    return _SHAPE


def make_nbest(n_utts: int = 7176, n_best: int = 10, seed: int = 0,
               min_len: int | None = None, max_len: int | None = None) -> SynthNbest:
    """AISHELL-1-test-shaped N-best lists.  With min_len/max_len the reference
    lengths are drawn uniformly from [min_len, max_len] instead (config 4:
    8..64)."""
    rng = np.random.default_rng(seed)
    ref_len, ref_edits = shape_table()
    stretched = min_len is not None or max_len is not None
    if stretched:
        lo, hi = min_len or 3, max_len or 37
        lens = rng.integers(lo, hi + 1, size=n_utts)
    else:
        lens = ref_len[np.arange(n_utts) % len(ref_len)]       # utterance order; config 1 = the first 100
    # Zipf-ish unigram distribution over N_DISTINCT_CHARS characters
    p = 1.0 / (np.arange(N_DISTINCT_CHARS) + 10.0)
    p /= p.sum()
    ed_vals = np.array(list(EDIT_HIST.keys()))
    ed_p = np.array(list(EDIT_HIST.values()), np.float64)
    ed_p /= ed_p.sum()
    gaps_mean = np.array([AM_GAP_MEAN[min(k, len(AM_GAP_MEAN) - 1)] if k < len(AM_GAP_MEAN) else 0.55
                          for k in range(max(n_best - 1, 1))])
    utt_ids, refs, hyps = [], [], []
    am = np.zeros((n_utts, n_best))
    edits = np.zeros((n_utts, n_best), np.int32)
    for u in range(n_utts):
        L = int(lens[u])
        ref_r = rng.choice(N_DISTINCT_CHARS, size=L, p=p)
        ref = [char_of_rank(int(r)) for r in ref_r]
        d = rng.choice(ed_vals, size=n_best, p=ed_p)
        if n_best > 10:
            d[10:] += 1
        if stretched:
            d = d[np.argsort(d + rng.uniform(0, 1.5, size=n_best), kind="stable")]
        else:                                   # the real per-(utterance, k) edit counts for k < 10
            d[:min(n_best, 10)] = ref_edits[u % len(ref_len), :min(n_best, 10)]
        hs = []
        for k in range(n_best):
            h = list(ref)
            for _ in range(int(d[k])):
                op = int(rng.integers(0, 3))
                if op == 0 and len(h) > 0:                       # substitution
                    h[int(rng.integers(0, len(h)))] = char_of_rank(int(rng.choice(N_DISTINCT_CHARS, p=p)))
                elif op == 1:                                    # insertion
                    h.insert(int(rng.integers(0, len(h) + 1)), char_of_rank(int(rng.choice(N_DISTINCT_CHARS, p=p))))
                elif len(h) > 1:                                 # deletion, keep length >= 1
                    del h[int(rng.integers(0, len(h)))]
            hs.append("".join(h))
        first = min(AM_FIRST_MAX, AM_FIRST_MAX - rng.gamma(shape=1.1, scale=(AM_FIRST_MAX - AM_FIRST_MEAN) / 1.1))
        g = rng.exponential(gaps_mean[:n_best - 1]) if n_best > 1 else np.zeros(0)
        am[u, 0] = first
        am[u, 1:] = first - np.cumsum(g)
        edits[u] = d
        utt_ids.append(f"SYN{u:07d}")
        refs.append("".join(ref))
        hyps.append(hs)
    return SynthNbest(utt_ids, refs, hyps, am, edits,
                      meta=dict(n_utts=n_utts, n_best=n_best, seed=seed, min_len=min_len, max_len=max_len))


def synthetic_lm_scores(nb: SynthNbest, seed: int = 1) -> np.ndarray:
    """lm = -9.96*L + N(0, 0.8) stand-in PLLs for combiner-only runs (config 5)."""
    rng = np.random.default_rng(seed)
    L = np.array([[len(h) for h in hs] for hs in nb.hyps], np.float64)
    return -9.96 * L + rng.normal(0.0, 0.8, size=L.shape)


def state_dict_keys(cfg: dict) -> List[str]:
    keys = ["bert.embeddings.word_embeddings.weight", "bert.embeddings.position_embeddings.weight",
            "bert.embeddings.token_type_embeddings.weight", "bert.embeddings.LayerNorm.weight",
            "bert.embeddings.LayerNorm.bias"]
    for i in range(cfg["num_layers"]):
        p = f"bert.encoder.layer.{i}."
        for m in ("attention.self.query", "attention.self.key", "attention.self.value", "attention.output.dense"):
            keys += [p + m + ".weight", p + m + ".bias"]
        keys += [p + "attention.output.LayerNorm.weight", p + "attention.output.LayerNorm.bias",
                 p + "intermediate.dense.weight", p + "intermediate.dense.bias",
                 p + "output.dense.weight", p + "output.dense.bias",
                 p + "output.LayerNorm.weight", p + "output.LayerNorm.bias"]
    keys += ["cls.predictions.bias", "cls.predictions.transform.dense.weight",
             "cls.predictions.transform.dense.bias", "cls.predictions.transform.LayerNorm.weight",
             "cls.predictions.transform.LayerNorm.bias", "cls.predictions.decoder.weight",
             "cls.predictions.decoder.bias"]
    return keys


def random_init_state_dict(cfg: dict, seed: int = 10, perturb: bool = False):
    """fp32 CPU state_dict with the HF BertForMaskedLM key names.

    perturb=False reproduces the distribution of HF's default init (what the
    north-star parity config uses).  perturb=True additionally randomises the
    biases and LayerNorm affine parameters so that bias / gamma / beta handling
    is actually exercised by the parity tests.
    """
    import torch

    g = torch.Generator().manual_seed(seed)
    H, I, V = cfg["hidden"], cfg["intermediate"], cfg["vocab"]
    shapes = {
        "bert.embeddings.word_embeddings.weight": (V, H),
        "bert.embeddings.position_embeddings.weight": (cfg["max_position"], H),
        "bert.embeddings.token_type_embeddings.weight": (cfg.get("type_vocab", 2), H),
    }
    sd = {}

    def normal(shape, std=0.02):
        return torch.empty(shape, dtype=torch.float32).normal_(0.0, std, generator=g)

    for k in state_dict_keys(cfg):
        if k in ("cls.predictions.decoder.weight", "cls.predictions.decoder.bias"):
            continue
        if k in shapes:
            sd[k] = normal(shapes[k])
        elif k.endswith("LayerNorm.weight"):
            sd[k] = 1.0 + normal((H,), 0.1) if perturb else torch.ones(H)
        elif k.endswith("LayerNorm.bias"):
            sd[k] = normal((H,), 0.1) if perturb else torch.zeros(H)
        elif k == "cls.predictions.bias":
            sd[k] = normal((V,), 0.5) if perturb else torch.zeros(V)
        elif k.endswith(".weight"):
            out_f, in_f = (I, H) if "intermediate.dense" in k else (H, I) if ".output.dense" in k and "attention" not in k else (H, H)
            sd[k] = normal((out_f, in_f))
        elif k.endswith(".bias"):
            n = I if "intermediate.dense" in k else H
            sd[k] = normal((n,), 0.05) if perturb else torch.zeros(n)
    sd["bert.embeddings.word_embeddings.weight"][PAD_ID].zero_()
    # tied exactly as in transformers (modeling_bert.py:915-918)
    sd["cls.predictions.decoder.weight"] = sd["bert.embeddings.word_embeddings.weight"]
    sd["cls.predictions.decoder.bias"] = sd["cls.predictions.bias"]
    return sd


def random_rescorebert_state_dict(cfg: dict, seed: int = 10, perturb: bool = False):
    """fp32 CPU state_dict of the reference's RescoreBert module (RescoreBert/model.py:7-11): the
    ``bert.*`` encoder of random_init_state_dict, a BertModel pooler (``bert.pooler.dense``) and
    ``linear.weight`` [1, H] / ``linear.bias`` [1], N(0, 0.02) / 0 (perturb: N(0, 0.5))."""
    import torch

    sd = {k: v for k, v in random_init_state_dict(cfg, seed, perturb).items() if k.startswith("bert.")}
    g = torch.Generator().manual_seed(seed + 1)
    H = cfg["hidden"]
    sd["bert.pooler.dense.weight"] = torch.empty(H, H).normal_(0.0, 0.02, generator=g)
    sd["bert.pooler.dense.bias"] = torch.zeros(H)
    sd["linear.weight"] = torch.empty(1, H).normal_(0.0, 0.02, generator=g)
    sd["linear.bias"] = torch.empty(1).normal_(0.0, 0.5, generator=g) if perturb else torch.zeros(1)
    return sd


def config_from_state_dict(sd) -> dict:
    """Infer the model shape from a BertForMaskedLM state_dict."""
    H = sd["bert.embeddings.word_embeddings.weight"].shape[1]
    n_layers = 0
    while f"bert.encoder.layer.{n_layers}.attention.self.query.weight" in sd:
        n_layers += 1
    return dict(num_layers=n_layers, hidden=H, num_heads=H // 64,
                intermediate=sd["bert.encoder.layer.0.intermediate.dense.weight"].shape[0],
                vocab=sd["bert.embeddings.word_embeddings.weight"].shape[0],
                max_position=sd["bert.embeddings.position_embeddings.weight"].shape[0],
                type_vocab=sd["bert.embeddings.token_type_embeddings.weight"].shape[0], ln_eps=1e-12)
