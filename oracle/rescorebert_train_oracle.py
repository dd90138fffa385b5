"""CPU restatement (plain torch fp32 + autograd) of RescoreBert distillation training.

TEST INFRASTRUCTURE ONLY — imported by tests/ and tools/; never by the product path.

Provenance.  The reference trains its RescoreBert student with RescoreBert/main.py on train_lm.json,
but that script is not in the reference tree (nor under baseline/_ref).  The formulas below are
therefore the contract of pllb_cls_train_* (include/pllb.h), pinned by this autograd restatement and
not by a reference golden:

  * model ....... BertModel -> last_hidden_state[:, 0, :] -> Linear(H, 1) (RescoreBert/model.py:13-21;
                  pll_oracle.bert_mlm_logits(..., return_hidden=True) is that BertModel forward)
  * MD .......... nn.MSELoss()(s, y): (1/B) sum_i (s_i - y_i)^2, y = teacher PLL
  * MWER ........ P = softmax over each utterance's rows of (am_weight * a + s);
                  (1/G) sum_g sum_{i in g} P_i (e_i - mean_g e), e = per-hypothesis CER
  * total ....... md_weight * MD + mwer_weight * MWER
  * optimizer ... torch.optim.AdamW over every parameter (weight decay 0.01 on all, linear.* too);
                  the pooler is a parameter that never receives a gradient, so AdamW skips it
  * [PAD] ....... the word-embedding lookup sends no gradient to row 0 (padding_idx)

Parity is defined at dropout 0, as for the MLM trainer (oracle/train_oracle.py).
"""
from __future__ import annotations

from typing import Dict, List

import numpy as np
import torch
import torch.nn.functional as F

from . import pll_oracle


def parameters(sd: Dict[str, torch.Tensor]) -> Dict[str, torch.Tensor]:
    """fp32 leaves of every tensor but position_ids (the pooler included)."""
    return {k: v.detach().clone().float().requires_grad_(True) for k, v in sd.items() if not k.endswith("position_ids")}


def scores(params, cfg, ids, mask) -> torch.Tensor:
    hid = pll_oracle.bert_mlm_logits(params, cfg, torch.as_tensor(ids, dtype=torch.long),
                                     torch.as_tensor(mask, dtype=torch.long), return_hidden=True, padding_idx=0)
    return F.linear(hid[:, 0, :], params["linear.weight"].reshape(1, -1), params["linear.bias"].reshape(1)).squeeze(-1)


def losses(s, target, am, err, group, md_weight=1.0, mwer_weight=0.0, am_weight=1.0):
    """(total, MD, MWER) as torch scalars; s is the score tensor (autograd flows through it)."""
    target, am, err = (torch.as_tensor(np.asarray(x), dtype=s.dtype) for x in (target, am, err))
    group = np.asarray(group)
    md = F.mse_loss(s, target)
    G = int(group[-1]) + 1
    mwer = s.new_zeros(())
    for g in range(G):
        idx = torch.as_tensor(np.nonzero(group == g)[0])
        p = torch.softmax(am_weight * am[idx] + s[idx], dim=0)
        mwer = mwer + (p * (err[idx] - err[idx].mean())).sum()
    mwer = mwer / G
    return md_weight * md + mwer_weight * mwer, md, mwer


def closed_form_dscore(s, target, am, err, group, md_weight=1.0, mwer_weight=0.0, am_weight=1.0) -> np.ndarray:
    """dL/ds in float64 from the closed forms the device's loss kernel evaluates:
    (2/B) md_weight (s_i - y_i) + (1/G) mwer_weight P_i (e_i - sum_{j in g} P_j e_j)."""
    s, target, am, err = (np.asarray(x, np.float64) for x in (s, target, am, err))
    group = np.asarray(group)
    B, G = len(s), int(group[-1]) + 1
    d = md_weight * 2.0 / B * (s - target)
    for g in range(G):
        idx = np.nonzero(group == g)[0]
        z = am_weight * am[idx] + s[idx]
        p = np.exp(z - z.max())
        p /= p.sum()
        d[idx] += mwer_weight / G * p * (err[idx] - (p * err[idx]).sum())
    return d


def loss_and_grads(sd, cfg, batch: dict, **weights):
    """One batch (a dict of RescoreBert/train.make_batches): (loss, scores, {name: grad}); parameters
    that receive no gradient (the pooler) are absent."""
    params = parameters(sd)
    s = scores(params, cfg, batch["input_ids"], batch["attention_mask"])
    loss, _, _ = losses(s, batch["target"], batch["am"], batch["err"], batch["group"], **weights)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in params.items() if p.grad is not None}
    return loss.item(), s.detach().numpy(), grads


def run_steps(params, cfg, batches: List[dict], lr: float, **weights) -> List[float]:
    """torch.optim.AdamW (defaults but lr) over `params`, one step per batch; returns the batch losses."""
    opt = torch.optim.AdamW(list(params.values()), lr=lr)
    out = []
    for b in batches:
        s = scores(params, cfg, b["input_ids"], b["attention_mask"])
        loss, _, _ = losses(s, b["target"], b["am"], b["err"], b["group"], **weights)
        loss.backward()
        opt.step()
        opt.zero_grad()
        out.append(loss.item())
    return out
