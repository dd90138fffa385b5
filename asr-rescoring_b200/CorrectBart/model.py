"""CorrectBart's one_hyp correction on the device.

The reference generates with ``BartForConditionalGeneration.generate(max_length=50)`` from the 1-best
hypothesis and scores the outputs with ``jiwer.cer`` (CorrectBart/compute_cer.py:8).  Here the model runs
through ``engine.Seq2SeqGenerator`` (greedy decoding, pllb_generate, or beam search, pllb_generate_beam,
when ``num_beams > 1``) and the CER through the Levenshtein kernel of ``cer_clients``."""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence

import numpy as np

from .. import engine
from ..tokenizer import encode_batch


class CorrectBart:
    """state_dict: a BartForConditionalGeneration state_dict (optionally under one module prefix);
    cfg: its BartConfig as a dict, which also supplies generate()'s settings (decoder_start_token_id,
    eos_token_id, pad_token_id, forced_bos_token_id, forced_eos_token_id); ``generation`` overrides them.
    tokenizer: a BertCharTokenizer (fnlp/bart-base-chinese uses BertTokenizer).  With ``num_beams > 1`` in
    the config or in ``generation``, correct() runs beam search (also reading num_return_sequences,
    length_penalty and early_stopping) and decodes the best hypothesis."""

    def __init__(self, state_dict, cfg: dict, tokenizer, device: int = 0, max_length: int = 50,
                 operand_dtype: str = "bf16", max_rows: int = 0, cls_id: int = 101, sep_id: int = 102,
                 generation: Optional[dict] = None):
        self.tokenizer = tokenizer
        self.cls_id, self.sep_id = cls_id, sep_id
        gen = dict(generation or {})
        self.beam = int(gen.get("num_beams", cfg.get("num_beams")) or 1) > 1
        settings = engine.beam_settings if self.beam else engine.generation_settings
        self.generation = settings(cfg, max_length=max_length, **gen)
        self.model = engine.Seq2SeqGenerator(state_dict, cfg, device=device, max_rows=max_rows,
                                             operand_dtype=operand_dtype, cls_id=cls_id, sep_id=sep_id)

    def close(self):
        self.model.close()

    def generate_packed(self, tokens: np.ndarray, offsets: np.ndarray, return_logits: bool = False):
        """Packed ids (no specials) -> (ids int32[n, max_length], lengths int32[n][, logits]); with beam
        search the best hypothesis of each sentence (no logits)."""
        if self.beam:
            if return_logits:
                raise ValueError("beam search returns hypothesis scores, not per-token logits")
            ids, lens, _ = self.model.beam_search_packed(tokens, offsets, self.generation)
            return ids[:, 0], lens[:, 0]
        return self.model.generate_packed(tokens, offsets, self.generation, return_logits=return_logits)

    def skip_ids(self) -> List[int]:
        g = self.generation
        return sorted({self.cls_id, self.sep_id, int(g["pad_token_id"]), int(g["decoder_start_token_id"]),
                       int(g["eos_token_id"])})

    def decode(self, ids: np.ndarray, lens: np.ndarray) -> List[str]:
        skip = self.skip_ids()
        return [self.tokenizer.decode(ids[i, :lens[i]], skip) for i in range(len(lens))]

    def correct(self, texts: Sequence[str]) -> List[str]:
        """One corrected sentence per input text."""
        if len(texts) == 0:
            return []
        tok, off = encode_batch(self.tokenizer, texts)
        ids, lens = self.generate_packed(tok, off)
        return self.decode(ids, lens)


def one_hyp(hyps_text: Dict[str, Dict[str, str]]) -> List[str]:
    """The one_hyp input: the 1-best (hyp_1) of every utterance, in utterance order."""
    return [hs["hyp_1"] for hs in hyps_text.values()]


def compute_cer(preds: Sequence[str], refs: Sequence[str]) -> float:
    """Corpus CER as jiwer.cer(refs, preds) computes it over lists: total edit distance over total
    reference characters (strings stripped, characters = code points)."""
    if len(preds) != len(refs):
        raise ValueError("prediction and reference lists differ in length")
    total = sum(len(r.strip()) for r in refs)
    if total == 0:
        raise ValueError("the references are empty")
    dist = engine.levenshtein(list(refs), list(preds))
    return float(np.asarray(dist, np.int64).sum()) / float(total)
