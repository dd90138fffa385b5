"""Text front end: hypothesis string -> wordpiece ids (SURVEY.md §8f rank 1).

The reference calls ``BertTokenizer.from_pretrained("bert-base-chinese").tokenize``
(MLM_PLL/preprocess.py:10,34).  That vocabulary is fetched from the HF hub at run time
and is not available offline, so two modes exist:

* ``BertCharTokenizer(vocab_file)``: BERT's BasicTokenizer + WordPiece restated for the
  case that matters here — every CJK character is its own token; runs of other
  characters are lower-cased, accent-stripped, split on punctuation and greedily
  longest-match wordpieced; unknown -> [UNK].  (transformers
  models/bert/tokenization_bert.py; checked against it in tests/test_host.py.)
* ``SyntheticCharTokenizer()``: deterministic char -> id map used with random-init
  weights (synth.synthetic_token_id).
"""
from __future__ import annotations

import unicodedata
from typing import Dict, List, Sequence, Tuple

import numpy as np

from .synth import UNK_ID, synthetic_token_id

TABLE_SIZE = 0x30000             # covers the BMP and every CJK extension block _is_cjk knows
TOK_SPACE, TOK_REMOVED, TOK_WORD = -1, -2, -3      # include/pllb.h PLLB_TOK_*


def _is_cjk(cp: int) -> bool:
    return (0x4E00 <= cp <= 0x9FFF or 0x3400 <= cp <= 0x4DBF or 0x20000 <= cp <= 0x2A6DF or
            0x2A700 <= cp <= 0x2B73F or 0x2B740 <= cp <= 0x2B81F or 0x2B820 <= cp <= 0x2CEAF or
            0xF900 <= cp <= 0xFAFF or 0x2F800 <= cp <= 0x2FA1F)


def _is_punct(ch: str) -> bool:
    cp = ord(ch)
    if 33 <= cp <= 47 or 58 <= cp <= 64 or 91 <= cp <= 96 or 123 <= cp <= 126:
        return True
    return unicodedata.category(ch).startswith("P")


def _is_control(ch: str) -> bool:
    if ch in ("\t", "\n", "\r"):
        return False
    return unicodedata.category(ch).startswith("C")


def _is_whitespace(ch: str) -> bool:
    return ch in (" ", "\t", "\n", "\r") or unicodedata.category(ch) == "Zs"


class SyntheticCharTokenizer:
    def tokenize(self, text: str) -> List[str]:
        return list(text)

    def convert_tokens_to_ids(self, tokens: List[str]) -> List[int]:
        return [synthetic_token_id(t) for t in tokens]

    def encode(self, text: str) -> List[int]:
        return self.convert_tokens_to_ids(self.tokenize(text))

    def char_table(self) -> np.ndarray:
        """Every code point is its own token (nothing is dropped)."""
        if getattr(self, "_table", None) is None:
            cp = np.arange(TABLE_SIZE, dtype=np.int64)
            rank = np.where((cp >= 0x4E00) & (cp < 0x4E00 + 20000), ((cp - 0x4E00) * 17143) % 20000, cp)
            self._table = (670 + rank % 7322).astype(np.int32)
        return self._table


class BertCharTokenizer:
    def __init__(self, vocab_file: str, do_lower_case: bool = True, unk_token: str = "[UNK]",
                 max_input_chars_per_word: int = 100):
        self.vocab: Dict[str, int] = {}
        with open(vocab_file, "r", encoding="utf-8") as f:
            for i, line in enumerate(f):
                self.vocab[line.rstrip("\n")] = i
        self.do_lower_case = do_lower_case
        self.unk_token = unk_token
        self.max_chars = max_input_chars_per_word

    # BasicTokenizer.tokenize
    def _basic(self, text: str) -> List[str]:
        out = []
        for ch in text:
            cp = ord(ch)
            if cp == 0 or cp == 0xFFFD or _is_control(ch):
                continue
            out.append(" " if _is_whitespace(ch) else ch)
        text = unicodedata.normalize("NFC", "".join(out))
        spaced = []
        for ch in text:
            spaced.append(f" {ch} " if _is_cjk(ord(ch)) else ch)
        words = []
        for tok in "".join(spaced).strip().split():
            if self.do_lower_case:
                tok = tok.lower()
                tok = "".join(c for c in unicodedata.normalize("NFD", tok) if unicodedata.category(c) != "Mn")
            cur = []
            for ch in tok:
                if _is_punct(ch):
                    if cur:
                        words.append("".join(cur))
                        cur = []
                    words.append(ch)
                else:
                    cur.append(ch)
            if cur:
                words.append("".join(cur))
        return " ".join(words).split()

    # WordpieceTokenizer.tokenize
    def _wordpiece(self, word: str) -> List[str]:
        if len(word) > self.max_chars:
            return [self.unk_token]
        pieces, start = [], 0
        while start < len(word):
            end, cur = len(word), None
            while start < end:
                sub = word[start:end]
                if start > 0:
                    sub = "##" + sub
                if sub in self.vocab:
                    cur = sub
                    break
                end -= 1
            if cur is None:
                return [self.unk_token]
            pieces.append(cur)
            start = end
        return pieces

    def tokenize(self, text: str) -> List[str]:
        return [p for w in self._basic(text) for p in self._wordpiece(w)]

    def convert_tokens_to_ids(self, tokens: List[str]) -> List[int]:
        unk = self.vocab.get(self.unk_token, UNK_ID)
        return [self.vocab.get(t, unk) for t in tokens]

    def encode(self, text: str) -> List[int]:
        return self.convert_tokens_to_ids(self.tokenize(text))

    def decode(self, ids: Sequence[int], skip_ids: Sequence[int] = (0, 101, 102)) -> str:
        """ids -> text for a character error rate: the ids in ``skip_ids`` (pass cls, sep, pad and the
        decoder's start / eos ids) are dropped, a ``##`` prefix is removed and the pieces are joined
        WITHOUT spaces.  (HF's decode puts a space between CJK tokens; jiwer.cer compares characters.)"""
        inv = getattr(self, "_inv", None)
        if inv is None:
            inv = self._inv = {i: t for t, i in self.vocab.items()}
        skip = set(int(i) for i in skip_ids)
        out = []
        for i in ids:
            i = int(i)
            if i in skip:
                continue
            t = inv.get(i, self.unk_token)
            out.append(t[2:] if t.startswith("##") else t)
        return "".join(out)

    def char_table(self) -> np.ndarray:
        """int32[TABLE_SIZE] for pllb_tokenize_host: the id of every character that BasicTokenizer
        always isolates as its own token (CJK ideographs, punctuation), TOK_SPACE / TOK_REMOVED for
        characters that emit nothing, TOK_WORD for everything whose tokenisation depends on its
        neighbours (those hypotheses go through ``encode``)."""
        if getattr(self, "_table", None) is not None:
            return self._table
        unk = self.vocab.get(self.unk_token, UNK_ID)
        table = np.full(TABLE_SIZE, TOK_WORD, np.int32)
        probe = next((chr(c) for c in range(0x4E00, 0x9FFF) if chr(c) in self.vocab), None)
        for cp in range(TABLE_SIZE):
            if 0xD800 <= cp <= 0xDFFF:
                continue
            ch = chr(cp)
            if cp == 0 or cp == 0xFFFD or _is_control(ch):
                table[cp] = TOK_REMOVED
            elif _is_whitespace(ch):
                table[cp] = TOK_SPACE
            elif _is_cjk(cp):
                n = unicodedata.normalize("NFC", ch)
                if len(n) == 1 and _is_cjk(ord(n)):
                    table[cp] = self.vocab.get(n, unk)
            elif _is_punct(ch):
                # context-free only if it stays one token between two ideographs
                one = self.encode(ch)
                if len(one) == 1 and (probe is None or
                                      self.encode(probe + ch + probe) == [self.vocab[probe], one[0], self.vocab[probe]]):
                    table[cp] = one[0]
        self._table = table
        return table


def encode_batch(tokenizer, strings: Sequence[str]) -> Tuple[np.ndarray, np.ndarray]:
    """All strings -> (ids int32[sum], offsets int64[n+1]): one pllb_tokenize_host call for the
    CJK/punctuation hypotheses, ``tokenizer.encode`` on the host for the flagged rest
    (replaces the per-sentence tokenizer calls of MLM_PLL/preprocess.py:10,16-27)."""
    from . import engine
    n = len(strings)
    cp, cp_off = engine.pack_strings(strings)
    ids, off, flag = engine.tokenize_packed(tokenizer.char_table(), cp, cp_off)
    if not flag.any():
        return ids, off
    lens = np.diff(off)
    host = {int(i): np.asarray(tokenizer.encode(strings[int(i)]), np.int32) for i in np.nonzero(flag)[0]}
    for i, v in host.items():
        lens[i] = len(v)
    new_off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=new_off[1:])
    out = np.empty(int(new_off[-1]), np.int32)
    keep = flag == 0
    shift = np.repeat(new_off[:-1][keep] - off[:-1][keep], np.diff(off)[keep])
    out[np.arange(len(ids), dtype=np.int64) + shift] = ids
    for i, v in host.items():
        out[new_off[i]:new_off[i + 1]] = v
    return out, new_off
