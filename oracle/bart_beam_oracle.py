"""fp32 CPU oracle of BART beam search (pllb_generate_beam, DESIGN.md §3.12).

* ``beam``: beam search written out over ``forward`` with the KV cache, restating items 1-9 of the
  contract in fp32; ``BeamSearch.select`` is one step on given logits (the replay test).  Every
  comparison records its margin: the 2K cut, the running K cut and order, the finished-merge cut and
  order, the early-stop test and the final order.  A CPU test shows ``beam`` equals
  ``generate(num_beams=K)`` token for token.
* ``hf_beam``: transformers' ``generate(num_beams=K)`` itself, for the comparisons.

The model helpers (``bart_config``, ``make_model``, ``encoder_inputs``, ``teacher_forced_logits``) are
those of ``bart_oracle``.
"""
from __future__ import annotations

import numpy as np

from .bart_oracle import _trim, encoder_inputs

DEAD = -1e8      # scores at or below this carry a -1e9 penalty: comparisons among them decide nothing


def _margin(a: float, b: float) -> float:
    if a <= DEAD and b <= DEAD:
        return float("inf")
    return float(a) - float(b)


def _order(vals, idx):
    """Positions of vals sorted by (value descending, index ascending)."""
    vals = np.asarray(vals, np.float32)
    return np.lexsort((np.asarray(idx), -vals.astype(np.float64)))


class BeamSearch:
    """State of beam search over n sentences x K beams (row i * K + b), fp32 as _beam_search computes it."""

    def __init__(self, n: int, gen: dict):
        self.n, self.K, self.ML = n, int(gen["num_beams"]), int(gen["max_length"])
        self.eos, self.pad, self.start = gen["eos_token_id"], gen["pad_token_id"], gen["decoder_start_token_id"]
        self.fb, self.fe = gen.get("forced_bos_token_id"), gen.get("forced_eos_token_id")
        self.lp = float(gen.get("length_penalty", 1.0))
        es = gen.get("early_stopping", False)
        self.es = "never" if isinstance(es, str) else bool(es)
        self.r = int(gen.get("num_return_sequences", 1))
        K, ML = self.K, self.ML
        self.run_seq = np.full((n * K, ML), self.pad, np.int64)
        self.run_seq[:, 0] = self.start
        self.run_score = np.tile(np.array([0.0] + [-1e9] * (K - 1), np.float32), n)
        self.fin_seq = self.run_seq.copy()
        self.fin_len = np.ones(n * K, np.int64)
        self.fin_score = np.full(n * K, -1e9, np.float32)
        self.fin_flag = np.zeros(n * K, bool)
        self.unsat = np.ones(n, bool)
        self.frozen = np.zeros(n, bool)
        self.margins = [[] for _ in range(n)]      # (t, kind, margin)
        self.parents, self.run_scores = [], []

    def _note(self, i, t, kind, m):
        self.margins[i].append((t, kind, float(m)))

    def select(self, logits, t: int):
        """Step t on fp32 logits [n * K, V] of the running beams."""
        import torch
        K, ML, V = self.K, self.ML, logits.shape[1]
        f32 = np.float32
        logp = torch.log_softmax(torch.as_tensor(logits, dtype=torch.float32), -1).numpy()
        forced = self.fe if (t == ML - 1 and self.fe is not None) else (self.fb if t == 1 else None)
        if forced is not None:
            logp = np.full_like(logp, -np.inf)
            logp[:, forced] = 0.0
        new_seq = self.run_seq.copy()
        parents = np.arange(self.n * K)
        for i in range(self.n):
            rows = slice(i * K, (i + 1) * K)
            if self.frozen[i]:
                new_seq[rows, t] = self.pad
                continue
            cand = (logp[rows] + self.run_score[rows, None]).astype(f32).ravel()
            # top 2K (+1 for the cut margin), ties to the lower flat index
            kth = -np.partition(-cand.astype(np.float64), 2 * K)[2 * K]
            pool = np.nonzero(cand >= kth)[0]
            pool = pool[_order(cand[pool], pool)][:2 * K + 1]
            top, val = pool[:2 * K], cand[pool[:2 * K]]
            self._note(i, t, "2K cut", _margin(cand[pool[2 * K - 1]], cand[pool[2 * K]]))
            beam_of, tok = top // V, top % V
            hit = (tok == self.eos) | (t == ML - 1)
            if hit[K - 1] or hit[K]:
                self._note(i, t, "K cut of the 2K", _margin(val[K - 1], val[K]))
            pen = np.where(hit, val + f32(-1e9), val).astype(f32)
            ro = _order(pen, np.arange(2 * K))
            self._note(i, t, "running cut", _margin(pen[ro[K - 1]], pen[ro[K]]))
            for k in range(K - 1):
                self._note(i, t, "running order", _margin(pen[ro[k]], pen[ro[k + 1]]))
            sel = ro[:K]
            par = i * K + beam_of[sel]
            # finished slots
            old_s, old_f = self.fin_score[rows].copy(), self.fin_flag[rows].copy()
            norm = f32(float(t) ** self.lp)
            fs = (val / norm).astype(f32)
            if old_f.all() and self.es is True:
                fs = (fs + f32(-1e9)).astype(f32)
            if not self.unsat[i]:
                fs = (fs + f32(-1e9)).astype(f32)
            jf = hit & (np.arange(2 * K) < K)
            fs = np.where(jf, fs, fs + f32(-1e9)).astype(f32)
            merged = np.concatenate([old_s, fs]).astype(f32)
            mo = _order(merged, np.arange(3 * K))
            self._note(i, t, "finished cut", _margin(merged[mo[K - 1]], merged[mo[K]]))
            for k in range(K - 1):
                self._note(i, t, "finished order", _margin(merged[mo[k]], merged[mo[k + 1]]))
            old_seq, old_len = self.fin_seq[rows].copy(), self.fin_len[rows].copy()
            for k, src in enumerate(mo[:K]):
                row = i * K + k
                if src < K:
                    self.fin_seq[row], self.fin_len[row] = old_seq[src], old_len[src]
                    self.fin_flag[row] = old_f[src]
                else:
                    c = src - K
                    self.fin_seq[row] = self.pad
                    self.fin_seq[row, :t] = self.run_seq[i * K + beam_of[c], :t]
                    self.fin_seq[row, t] = tok[c]
                    self.fin_len[row] = t + 1
                    self.fin_flag[row] = jf[c]
                self.fin_score[row] = merged[src]
            # running beams
            new_seq[rows, :t] = self.run_seq[par, :t]
            new_seq[rows, t] = tok[sel]
            self.run_score[rows] = pen[sel]
            parents[rows] = par
            # early-stop heuristic after the step, then freezing
            L = ML - 1 if (self.es == "never" and self.lp > 0) else t
            best = f32(pen[sel[0]] / f32(float(L) ** self.lp))
            fsc, ffl = self.fin_score[rows], self.fin_flag[rows]
            mn = fsc.min()
            worst = np.where(ffl, mn, f32(-1e9))
            for w in worst:
                if w > DEAD:
                    self._note(i, t, "early-stop test", abs(float(best) - float(w)))
            self.unsat[i] = self.unsat[i] and bool((best > worst).any())
            if not self.unsat[i] or (self.es is True and ffl.all()):
                self.frozen[i] = True
        self.run_seq = new_seq
        self.parents.append(parents)
        self.run_scores.append(self.run_score.copy())
        return parents

    def done(self, t: int) -> bool:
        return bool(self.frozen.all()) or t >= self.ML - 1

    def result(self):
        """(ids [n, r, ML] padded with pad, lengths [n, r], scores [n, r]); notes the final-order margins."""
        n, K, r, ML = self.n, self.K, self.r, self.ML
        ids = np.full((n, r, ML), self.pad, np.int64)
        lens = np.zeros((n, r), np.int64)
        sc = np.zeros((n, r), np.float32)
        for i in range(n):
            for k in range(r):
                row = i * K + k
                lens[i, k] = self.fin_len[row]
                ids[i, k, :lens[i, k]] = self.fin_seq[row, :lens[i, k]]
                sc[i, k] = self.fin_score[row]
            s = self.fin_score[i * K:(i + 1) * K]
            for k in range(min(r, K - 1)):
                self._note(i, ML, "final order", _margin(s[k], s[k + 1]))
        return ids, lens, sc

    def min_margin(self, i: int, scale=None) -> float:
        """Smallest margin of sentence i; with scale(t) each margin is divided by it first."""
        ms = [m / (scale(t) if scale else 1.0) for t, _, m in self.margins[i]]
        return min(ms) if ms else float("inf")


def beam(model, sents, cls_id, sep_id, gen: dict) -> BeamSearch:
    """Beam search over forward with the KV cache; gen holds generation_settings keys plus num_beams,
    num_return_sequences, length_penalty and early_stopping.  Returns the BeamSearch after the run
    (``result()`` gives ids / lengths / scores, ``margins`` the decisions)."""
    import torch
    ids, mask = encoder_inputs(sents, cls_id, sep_id)
    n, K = len(sents), int(gen["num_beams"])
    bs = BeamSearch(n, gen)
    with torch.no_grad():
        enc = model.get_encoder()(input_ids=ids, attention_mask=mask)
        enc.last_hidden_state = enc.last_hidden_state.repeat_interleave(K, 0)
        mask_k = mask.repeat_interleave(K, 0)
        past = None
        for t in range(1, bs.ML):
            cur = torch.tensor(bs.run_seq[:, t - 1:t])
            o = model(encoder_outputs=enc, attention_mask=mask_k, decoder_input_ids=cur, past_key_values=past,
                      use_cache=True)
            par = bs.select(o.logits[:, -1].float().numpy(), t)
            past = o.past_key_values
            past.reorder_cache(torch.as_tensor(par, dtype=torch.long))
            if bs.done(t):
                break
    return bs


def hf_beam(model, sents, cls_id, sep_id, gen: dict):
    """generate(num_beams=K, num_return_sequences=K, output_scores=True): per sentence the K hypotheses
    (ids up to and including EOS) and their sequences_scores."""
    import torch
    ids, mask = encoder_inputs(sents, cls_id, sep_id)
    K = int(gen["num_beams"])
    with torch.no_grad():
        out = model.generate(input_ids=ids, attention_mask=mask, num_beams=K, num_return_sequences=K, do_sample=False,
                             max_length=gen["max_length"], decoder_start_token_id=gen["decoder_start_token_id"],
                             eos_token_id=gen["eos_token_id"], pad_token_id=gen["pad_token_id"],
                             forced_bos_token_id=gen.get("forced_bos_token_id"),
                             forced_eos_token_id=gen.get("forced_eos_token_id"), min_length=0,
                             no_repeat_ngram_size=0, repetition_penalty=1.0,
                             length_penalty=float(gen.get("length_penalty", 1.0)),
                             early_stopping=gen.get("early_stopping", False),
                             output_scores=True, return_dict_in_generate=True)
    seqs = [_trim(r, gen["eos_token_id"]) for r in out.sequences.tolist()]
    sc = out.sequences_scores.float().numpy()
    return [[seqs[i * K + k] for k in range(K)] for i in range(len(sents))], sc.reshape(len(sents), K)
