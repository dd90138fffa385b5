"""fp32 CPU oracle of greedy BART generation (pllb_generate, DESIGN.md §3.11).

* ``make_model``: a random-init ``transformers.BartForConditionalGeneration`` (post-LN, gelu) whose
  biases, LayerNorm affines and ``final_logits_bias`` are randomised too, so every one of them is
  exercised.
* ``greedy``: the greedy loop written out over ``forward`` with the KV cache: the argmax of
  ``logits[:, -1]``, forced BOS / EOS, pad after EOS, stop when all rows finished or at max_length.
  A CPU test shows it equals ``generate(num_beams=1, do_sample=False)`` token for token.
* ``teacher_forced_logits``: the full fp32 logits at every position of a given decoder sequence.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np


def bart_config(d_model=256, layers=2, ffn=1024, vocab=8000, max_position=128, scale_embedding=False, init_std=0.1,
                **kw):
    """init_std 0.1 (HF: 0.02): with 0.02 the tied embeddings dominate and every sentence repeats its start token."""
    from transformers import BartConfig
    return BartConfig(vocab_size=vocab, d_model=d_model, encoder_layers=layers, decoder_layers=layers,
                      encoder_attention_heads=d_model // 64, decoder_attention_heads=d_model // 64,
                      encoder_ffn_dim=ffn, decoder_ffn_dim=ffn, max_position_embeddings=max_position,
                      activation_function="gelu", scale_embedding=scale_embedding, dropout=0.0,
                      attention_dropout=0.0, activation_dropout=0.0, pad_token_id=0, bos_token_id=101,
                      eos_token_id=102, decoder_start_token_id=102, forced_bos_token_id=None,
                      forced_eos_token_id=None, init_std=init_std, **kw)


def make_model(config, seed: int = 0, perturb: bool = True):
    import torch
    from transformers import BartForConditionalGeneration
    torch.manual_seed(seed)
    m = BartForConditionalGeneration(config).eval()
    if perturb:
        g = torch.Generator().manual_seed(seed + 1)
        with torch.no_grad():
            for name, p in m.named_parameters():
                if name.endswith(".bias"):
                    p.copy_(0.02 * torch.randn(p.shape, generator=g))
                elif "layer_norm" in name or "layernorm" in name:
                    p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g))
            m.final_logits_bias.copy_(0.1 * torch.randn(m.final_logits_bias.shape, generator=g))
    return m


def encoder_inputs(sents: Sequence[Sequence[int]], cls_id: int, sep_id: int, pad_id: int = 0):
    """[CLS] t [SEP], right-padded, with the attention mask."""
    import torch
    T = max(len(s) for s in sents) + 2
    ids = torch.full((len(sents), T), pad_id, dtype=torch.long)
    mask = torch.zeros((len(sents), T), dtype=torch.long)
    for i, s in enumerate(sents):
        row = [cls_id] + list(s) + [sep_id]
        ids[i, :len(row)] = torch.tensor(row)
        mask[i, :len(row)] = 1
    return ids, mask


def hf_generate(model, sents, cls_id, sep_id, gen: dict) -> List[List[int]]:
    """model.generate() with the greedy settings, per sentence the ids up to and including EOS."""
    import torch
    ids, mask = encoder_inputs(sents, cls_id, sep_id)
    with torch.no_grad():
        out = model.generate(input_ids=ids, attention_mask=mask, num_beams=1, do_sample=False,
                             max_length=gen["max_length"], decoder_start_token_id=gen["decoder_start_token_id"],
                             eos_token_id=gen["eos_token_id"], pad_token_id=gen["pad_token_id"],
                             forced_bos_token_id=gen.get("forced_bos_token_id"),
                             forced_eos_token_id=gen.get("forced_eos_token_id"), min_length=0,
                             no_repeat_ngram_size=0, repetition_penalty=1.0)
    return [_trim(r, gen["eos_token_id"]) for r in out.tolist()]


def _trim(row, eos):
    for j in range(1, len(row)):
        if row[j] == eos:
            return row[:j + 1]
    return row


def greedy(model, sents, cls_id, sep_id, gen: dict):
    """(ids int64[n, max_length] padded with pad, lengths int64[n], chosen-token logits float32[n, max_length])."""
    import torch
    ids, mask = encoder_inputs(sents, cls_id, sep_id)
    n, ML = len(sents), int(gen["max_length"])
    eos, pad = gen["eos_token_id"], gen["pad_token_id"]
    fb, fe = gen.get("forced_bos_token_id"), gen.get("forced_eos_token_id")
    out = np.full((n, ML), pad, np.int64)
    out[:, 0] = gen["decoder_start_token_id"]
    lens = np.zeros(n, np.int64)
    logit = np.zeros((n, ML), np.float32)
    with torch.no_grad():
        enc = model.get_encoder()(input_ids=ids, attention_mask=mask)
        past = None
        cur = torch.tensor(out[:, :1])
        for t in range(1, ML):
            o = model(encoder_outputs=enc, attention_mask=mask, decoder_input_ids=cur, past_key_values=past,
                      use_cache=True)
            past = o.past_key_values
            lg = o.logits[:, -1].float()
            choice = lg.argmax(-1)
            forced = fe if (t == ML - 1 and fe is not None) else (fb if t == 1 else None)
            if forced is not None:
                choice = torch.full_like(choice, forced)
            val = lg.gather(1, choice[:, None])[:, 0]
            for i in range(n):
                if lens[i] > 0:
                    out[i, t] = pad
                    continue
                out[i, t] = int(choice[i])
                logit[i, t] = float(val[i])
                if out[i, t] == eos or t == ML - 1:
                    lens[i] = t + 1
            cur = torch.tensor(out[:, t:t + 1])
            if (lens > 0).all():
                break
    lens[lens == 0] = ML
    return out, lens, logit


def teacher_forced_logits(model, sent: Sequence[int], dec: Sequence[int], cls_id: int, sep_id: int) -> np.ndarray:
    """fp32 logits [len(dec), vocab]; row j is the distribution over the token at position j + 1."""
    import torch
    ids, mask = encoder_inputs([sent], cls_id, sep_id)
    with torch.no_grad():
        o = model(input_ids=ids, attention_mask=mask, decoder_input_ids=torch.tensor([list(dec)]), use_cache=False)
    return o.logits[0].float().numpy()
