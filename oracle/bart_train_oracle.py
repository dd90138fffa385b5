"""fp32 CPU oracle of one CorrectBart training step (pllb_s2s_train_*, DESIGN.md §3.13).

``step`` runs transformers' ``BartForConditionalGeneration.forward(input_ids, attention_mask, labels=labels)``
in train mode at dropout 0, ``loss.backward()`` and one ``torch.optim.AdamW`` step over ``model.parameters()``,
all in fp32 on the host.  It returns the loss, the per-position losses (0 where the label is -100), the
gradients under state_dict keys (a tied tensor once, under ``model.shared.weight``) and the updated weights.
"""
from __future__ import annotations

from typing import Dict, Optional

import numpy as np


def token_losses(logits, labels) -> np.ndarray:
    """-log_softmax(logits)[label] per position, 0 where the label is -100 ([B, T_dec] float32)."""
    import torch
    lab = torch.as_tensor(np.asarray(labels), dtype=torch.long)
    ce = torch.nn.functional.cross_entropy(logits.float().reshape(-1, logits.shape[-1]), lab.reshape(-1),
                                           ignore_index=-100, reduction="none")
    return ce.reshape(lab.shape).detach().numpy().astype(np.float32)


def _grads(model) -> Dict[str, "torch.Tensor"]:
    """Gradients under state_dict keys; a parameter reachable under several names (tied) appears once, under the
    first of them, which for BART's shared table is ``model.shared.weight``."""
    return {n: (p.grad.detach().clone() if p.grad is not None else p.detach().new_zeros(p.shape))
            for n, p in model.named_parameters()}


def step(model, input_ids, attention_mask, labels, lr: float = 1e-5, betas=(0.9, 0.999), eps: float = 1e-8,
         weight_decay: float = 0.01, optimizer: Optional["torch.optim.Optimizer"] = None, update: bool = True):
    """One training step of ``model`` (modified in place when ``update``).  Pass the same ``optimizer`` to later
    calls to continue one AdamW run; a fresh one is created otherwise.  Returns (loss, token losses [B, T_dec],
    grads {name: tensor}, optimizer)."""
    import torch
    model.train()
    if optimizer is None:
        optimizer = torch.optim.AdamW(model.parameters(), lr=lr, betas=betas, eps=eps, weight_decay=weight_decay)
    optimizer.zero_grad(set_to_none=True)
    out = model(input_ids=torch.as_tensor(np.asarray(input_ids), dtype=torch.long),
                attention_mask=torch.as_tensor(np.asarray(attention_mask), dtype=torch.long),
                labels=torch.as_tensor(np.asarray(labels), dtype=torch.long))
    out.loss.backward()
    tl = token_losses(out.logits.detach(), labels)
    grads = _grads(model)
    if update:
        optimizer.step()
    return float(out.loss.detach()), tl, grads, optimizer


def train_epochs(model, batches, epochs: int, lr: float, weight_decay: float = 0.01):
    """The oracle of CorrectBart/train.py's loop: one AdamW for the run, batches in order, mean batch loss per
    epoch.  ``batches``: dicts with input_ids / attention_mask / labels."""
    import torch
    opt = torch.optim.AdamW(model.parameters(), lr=lr, weight_decay=weight_decay)
    losses = []
    for _ in range(epochs):
        tot = 0.0
        for b in batches:
            loss, _, _, _ = step(model, b["input_ids"], b["attention_mask"], b["labels"], optimizer=opt)
            tot += loss
        losses.append(tot / max(len(batches), 1))
    return losses
