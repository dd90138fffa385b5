"""Host-side driver of libpllb200.so: weight handoff, PLL scoring, Levenshtein, λ-sweep.

PyTorch is used only to own device memory (weights on their way in, caller-visible
outputs) and for the current CUDA stream; all arithmetic happens in the library.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional, Sequence

import numpy as np

from . import _lib
from ._lib import ClsLossDesc, LayerWeights, ModelDesc, Stats, TrainDesc, Weights, check

VARIANTS = {"B": 0, "A": 1, "C": 2, 0: 0, 1: 1, 2: 2}
OPERAND_DTYPES = {"bf16": 0, "fp16": 1, "bf16+fp16head": 2, "bf16+fp16tail": 3}   # pllb_model_desc.operand_dtype


def operand_dtype_code(name: str) -> int:
    """"bf16" | "fp16" | "bf16+fp16head" (bf16 encoder, fp16 MLM head) | "bf16+fp16tail" (bf16 for the
    first half of the encoder layers, fp16 for the second half and the head) | "fp16from:K" (bf16 for
    layers < K, fp16 for layers >= K and the head)."""
    if name.startswith("fp16from:"):
        return 16 + int(name.split(":", 1)[1])
    return OPERAND_DTYPES[name]
# bf16 operands on every encoder GEMM and attention MMA (98.9 % of the FLOPs), IEEE fp16 operands on the
# two MLM-head GEMMs: same speed as all-bf16 (measured), and the largest single rounding site is gone
DEFAULT_OPERAND_DTYPE = "bf16+fp16head"
GEMM_KINDS = ("qkv", "attn_out", "ffn1", "ffn2", "head_transform", "decoder_lse")


def _np_ptr(a: np.ndarray):
    return ctypes.c_void_p(a.ctypes.data)


def weights_struct(get, num_layers: int, keys):
    """pllb_weights over the tensors ``get(key)`` returns (CUDA fp32, contiguous) for the HF
    BertForMaskedLM state_dict names.  Returns (struct, list keeping the tensors and the layer array
    alive).  The MLM head is optional: a RescoreBert checkpoint (BertModel + Linear(H, 1)) has none."""
    keys = set(keys)
    keep = []

    def dp(key):
        t = get(key)
        keep.append(t)
        return ctypes.c_void_p(t.data_ptr())

    layers = (LayerWeights * max(num_layers, 1))()
    keep.append(layers)
    for i in range(num_layers):
        p = f"bert.encoder.layer.{i}."
        lw = layers[i]
        lw.q_w, lw.q_b = dp(p + "attention.self.query.weight"), dp(p + "attention.self.query.bias")
        lw.k_w, lw.k_b = dp(p + "attention.self.key.weight"), dp(p + "attention.self.key.bias")
        lw.v_w, lw.v_b = dp(p + "attention.self.value.weight"), dp(p + "attention.self.value.bias")
        lw.ao_w, lw.ao_b = dp(p + "attention.output.dense.weight"), dp(p + "attention.output.dense.bias")
        lw.ao_ln_g, lw.ao_ln_b = dp(p + "attention.output.LayerNorm.weight"), dp(p + "attention.output.LayerNorm.bias")
        lw.ff1_w, lw.ff1_b = dp(p + "intermediate.dense.weight"), dp(p + "intermediate.dense.bias")
        lw.ff2_w, lw.ff2_b = dp(p + "output.dense.weight"), dp(p + "output.dense.bias")
        lw.out_ln_g, lw.out_ln_b = dp(p + "output.LayerNorm.weight"), dp(p + "output.LayerNorm.bias")
    w = Weights()
    w.word_emb = dp("bert.embeddings.word_embeddings.weight")
    w.pos_emb = dp("bert.embeddings.position_embeddings.weight")
    w.type_emb = dp("bert.embeddings.token_type_embeddings.weight")
    w.emb_ln_g = dp("bert.embeddings.LayerNorm.weight")
    w.emb_ln_b = dp("bert.embeddings.LayerNorm.bias")
    w.layers = ctypes.cast(layers, ctypes.POINTER(LayerWeights))
    if "cls.predictions.transform.dense.weight" in keys:
        w.head_w = dp("cls.predictions.transform.dense.weight")
        w.head_b = dp("cls.predictions.transform.dense.bias")
        w.head_ln_g = dp("cls.predictions.transform.LayerNorm.weight")
        w.head_ln_b = dp("cls.predictions.transform.LayerNorm.bias")
        w.decoder_w = dp("cls.predictions.decoder.weight" if "cls.predictions.decoder.weight" in keys
                         else "bert.embeddings.word_embeddings.weight")
        w.decoder_b = dp("cls.predictions.bias" if "cls.predictions.bias" in keys else "cls.predictions.decoder.bias")
    return w, keep


def _model_desc(cfg: dict, operand_dtype: int = 0, cls_id: int = 101, sep_id: int = 102, mask_id: int = 103) -> ModelDesc:
    return ModelDesc(cfg["num_layers"], cfg["hidden"], cfg["num_heads"], cfg["intermediate"], cfg["vocab"],
                     cfg["max_position"], float(cfg.get("ln_eps", 1e-12)), cls_id, sep_id, mask_id, operand_dtype)


class _Handle:
    """Owner of one library handle ``self._h``, released by the symbol ``_DESTROY`` names."""

    _DESTROY = ""

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            getattr(self._lib, self._DESTROY)(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class PllScorer(_Handle):
    """BERT masked-LM pseudo-log-likelihood scorer; stands in for the
    ``BertForMaskedLM`` + ``run_one_epoch(do_scoring=True)`` pair of
    MLM_PLL/main.py:73-114,184-187."""

    _DESTROY = "pllb_destroy"

    def __init__(self, state_dict: Dict[str, "torch.Tensor"], cfg: Optional[dict] = None, device: int = 0,
                 max_chunk_tokens: int = 0, cls_id: int = 101, sep_id: int = 102, mask_id: int = 103,
                 operand_dtype: str = DEFAULT_OPERAND_DTYPE):
        import torch
        from .synth import config_from_state_dict

        self._lib = _lib.load()
        _lib.require_device()
        self._h = ctypes.c_void_p()
        self.cfg = dict(cfg) if cfg is not None else config_from_state_dict(state_dict)
        self.device = device
        dev = torch.device("cuda", device)
        nl = self.cfg["num_layers"]
        w, keep = weights_struct(lambda key: state_dict[key].detach().to(device=dev, dtype=torch.float32).contiguous(),
                                 nl, state_dict.keys())
        self.has_mlm_head = bool(w.head_w)
        d = _model_desc(self.cfg, operand_dtype_code(operand_dtype), cls_id, sep_id, mask_id)
        self.operand_dtype = operand_dtype
        torch.cuda.synchronize(dev)
        check(self._lib.pllb_create(ctypes.byref(self._h), ctypes.byref(d), ctypes.byref(w), int(max_chunk_tokens), device))
        del keep   # the library made its own (bf16 / fp32) copies

    # ------------------------------------------------------------------ scoring
    @staticmethod
    def _check_packed(tokens, offsets):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        if offsets.ndim != 1 or len(offsets) < 1:
            raise ValueError("offsets must be a 1-D array of n_hyp+1 entries")
        return offsets

    def score_packed(self, tokens: np.ndarray, offsets: np.ndarray, return_token_logp: bool = False):
        """HOST arrays in, HOST arrays out (H2D + score + D2H inside one C call).
        tokens: int32 wordpiece ids of all hypotheses back to back (no specials);
        offsets: int64[n_hyp+1].  Returns float64[n_hyp] PLLs (and float32 per-token terms)."""
        offsets = self._check_packed(tokens, offsets)
        tokens = np.ascontiguousarray(tokens, dtype=np.int32)
        n = len(offsets) - 1
        out = np.zeros(n, np.float64)
        tl = np.zeros(int(offsets[-1]), np.float32) if return_token_logp else None
        check(self._lib.pllb_score_host(self._h, _np_ptr(tokens), _np_ptr(offsets), n, _np_ptr(out),
                                        _np_ptr(tl) if tl is not None else None))
        return (out, tl) if return_token_logp else out

    def score_device(self, tokens_cuda, offsets: np.ndarray, out=None, token_logp=None):
        """tokens_cuda: torch int32 CUDA tensor; offsets: host int64.  Asynchronous on the
        current torch stream; returns a torch float64 CUDA tensor [n_hyp]."""
        import torch
        offsets = self._check_packed(None, offsets)
        n = len(offsets) - 1
        assert tokens_cuda.is_cuda and tokens_cuda.dtype == torch.int32 and tokens_cuda.is_contiguous()
        if out is None:
            out = torch.zeros(n, dtype=torch.float64, device=tokens_cuda.device)
        stream = torch.cuda.current_stream(tokens_cuda.device).cuda_stream
        check(self._lib.pllb_score(self._h, ctypes.c_void_p(tokens_cuda.data_ptr()), _np_ptr(offsets), n,
                                   ctypes.c_void_p(out.data_ptr()),
                                   ctypes.c_void_p(token_logp.data_ptr()) if token_logp is not None else None,
                                   ctypes.c_void_p(stream)))
        return out

    def score_cls_packed(self, tokens: np.ndarray, offsets: np.ndarray, linear_w, linear_b: float) -> np.ndarray:
        """Sequence-level scores (RescoreBert/model.py:13-21): every hypothesis runs through the
        encoder once as [CLS] t [SEP]; returns float32[n_hyp] = Linear(H,1)([CLS] state)."""
        offsets = self._check_packed(tokens, offsets)
        tokens = np.ascontiguousarray(tokens, dtype=np.int32)
        lw = np.ascontiguousarray(np.asarray(linear_w, np.float32).reshape(-1))
        if lw.shape[0] != self.cfg["hidden"]:
            raise ValueError("linear_w must have `hidden` elements")
        n = len(offsets) - 1
        out = np.zeros(n, np.float32)
        check(self._lib.pllb_score_cls_host(self._h, _np_ptr(tokens), _np_ptr(offsets), n, _np_ptr(lw),
                                            float(linear_b), _np_ptr(out)))
        return out

    def score_hyps(self, hyps: Dict[str, Dict[str, Sequence[int]]]) -> Dict[str, Dict[str, float]]:
        """{utt: {hyp: [token ids]}} -> {utt: {hyp: PLL}}; a hypothesis with no tokens keeps
        the int 0 of the reference's skeleton (MLM_PLL/main.py:189-193)."""
        flat, off = [], [0]
        for hs in hyps.values():
            for toks in hs.values():
                flat.extend(toks)
                off.append(len(flat))
        pll = self.score_packed(np.asarray(flat, np.int32), np.asarray(off, np.int64))
        out, i = {}, 0
        for u, hs in hyps.items():
            out[u] = {}
            for h, toks in hs.items():
                out[u][h] = float(pll[i]) if len(toks) > 0 else 0
                i += 1
        return out

    # ------------------------------------------------------------------ BERTScore (RMBR)
    def embed(self, tokens_cuda, offsets: np.ndarray, num_layers: int, out=None):
        """fp32 hidden states after ``num_layers`` encoder layers (0 = embedding LayerNorm) of every
        hypothesis as [CLS] t [SEP] (pllb_embed).  tokens_cuda: torch int32 CUDA tensor (no specials);
        offsets: host int64[n+1].  Returns a torch float32 CUDA tensor [sum (L+2), hidden]; sequence i
        starts at row offsets[i] - offsets[0] + 2 i.  Asynchronous on the current torch stream."""
        import torch
        offsets = self._check_packed(None, offsets)
        n = len(offsets) - 1
        rows = int(offsets[-1] - offsets[0]) + 2 * n
        assert tokens_cuda.is_cuda and tokens_cuda.dtype == torch.int32 and tokens_cuda.is_contiguous()
        if out is None:
            out = torch.empty(max(rows, 1), self.cfg["hidden"], dtype=torch.float32, device=tokens_cuda.device)
        elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() < rows * self.cfg["hidden"]:
            raise ValueError("out must be a contiguous float32 CUDA tensor of at least [rows, hidden]")
        stream = torch.cuda.current_stream(tokens_cuda.device).cuda_stream
        check(self._lib.pllb_embed(self._h, ctypes.c_void_p(tokens_cuda.data_ptr()), _np_ptr(offsets), n, int(num_layers),
                                   ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)))
        return out[:rows]

    def bertscore(self, emb, row_off: np.ndarray, cand: np.ndarray, ref: np.ndarray, out=None):
        """BERTScore recall R(cand[p], ref[p]) of every pair (pllb_bertscore).  emb: torch float32 CUDA
        [rows, hidden] (what :meth:`embed` returns); row_off: host int64[n_seq+1] row ranges of the
        sequences; cand / ref: host int32[n_pairs] sequence indices, best grouped by candidate.
        Returns a torch float32 CUDA tensor [n_pairs].  Asynchronous on the current torch stream."""
        import torch
        row_off = np.ascontiguousarray(row_off, np.int64)
        cand = np.ascontiguousarray(cand, np.int32)
        ref = np.ascontiguousarray(ref, np.int32)
        if row_off.ndim != 1 or len(row_off) < 1 or cand.shape != ref.shape or cand.ndim != 1:
            raise ValueError("row_off must be int64[n_seq+1], cand and ref equal int32[n_pairs]")
        if not (emb.is_cuda and emb.dtype == torch.float32 and emb.is_contiguous() and emb.shape[-1] == self.cfg["hidden"]):
            raise ValueError("emb must be a contiguous float32 CUDA tensor [rows, hidden]")
        if len(row_off) > 1 and row_off[-1] > emb.shape[0]:
            raise ValueError("row_off reaches past the rows of emb")
        if out is None:
            out = torch.empty(len(cand), dtype=torch.float32, device=emb.device)
        stream = torch.cuda.current_stream(emb.device).cuda_stream
        check(self._lib.pllb_bertscore(self._h, ctypes.c_void_p(emb.data_ptr()), _np_ptr(row_off), len(row_off) - 1,
                                       _np_ptr(cand), _np_ptr(ref), len(cand), ctypes.c_void_p(out.data_ptr()),
                                       ctypes.c_void_p(stream)))
        return out

    # ------------------------------------------------------------------ parity hooks
    def expand(self, tokens: np.ndarray, offsets: np.ndarray):
        import torch
        offsets = self._check_packed(tokens, offsets)
        L = np.diff(offsets)
        dev = torch.device("cuda", self.device)
        t = torch.from_numpy(np.ascontiguousarray(tokens, np.int32)).to(dev)
        ids = torch.zeros(max(int((L * (L + 2)).sum()), 1), dtype=torch.int32, device=dev)
        mp = torch.zeros(max(int(L.sum()), 1), dtype=torch.int32, device=dev)
        lab = torch.zeros_like(mp)
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(self._lib.pllb_expand(self._h, ctypes.c_void_p(t.data_ptr()), _np_ptr(offsets), len(L),
                                    ctypes.c_void_p(ids.data_ptr()), ctypes.c_void_p(mp.data_ptr()),
                                    ctypes.c_void_p(lab.data_ptr()), ctypes.c_void_p(stream)))
        torch.cuda.synchronize(dev)
        return (ids.cpu().numpy()[:int((L * (L + 2)).sum())], mp.cpu().numpy()[:int(L.sum())],
                lab.cpu().numpy()[:int(L.sum())])

    def hidden(self, tokens: np.ndarray, offsets: np.ndarray, upto_layer: int):
        import torch
        offsets = self._check_packed(tokens, offsets)
        L = np.diff(offsets)
        rows = int((L * (L + 2)).sum())
        dev = torch.device("cuda", self.device)
        t = torch.from_numpy(np.ascontiguousarray(tokens, np.int32)).to(dev)
        out = torch.zeros(max(rows, 1), self.cfg["hidden"], dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        check(self._lib.pllb_debug_hidden(self._h, ctypes.c_void_p(t.data_ptr()), _np_ptr(offsets), len(L), upto_layer,
                                          ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)))
        torch.cuda.synchronize(dev)
        return out[:rows].cpu()

    # ------------------------------------------------------------------ stats
    def set_timing(self, enable: bool):
        check(self._lib.pllb_set_timing(self._h, int(enable)))

    def reset_stats(self):
        check(self._lib.pllb_reset_stats(self._h))

    def stats(self) -> dict:
        s = Stats()
        check(self._lib.pllb_get_stats(self._h, ctypes.byref(s)))
        ms = (ctypes.c_float * 6)()
        fl = (ctypes.c_double * 6)()
        check(self._lib.pllb_get_gemm_breakdown(self._h, ms, fl))
        d = {n: getattr(s, n) for n, _ in Stats._fields_}
        d["gemm_ms_by_kind"] = dict(zip(GEMM_KINDS, [float(x) for x in ms]))
        d["gemm_flops_by_kind"] = dict(zip(GEMM_KINDS, [float(x) for x in fl]))
        d["workspace_bytes"] = int(self._lib.pllb_workspace_bytes(self._h))
        return d


def _prefix_lengths(attention_mask, shape) -> np.ndarray:
    am = np.asarray(attention_mask)
    if am.shape != shape:
        raise ValueError("input_ids and attention_mask must be equal [B, T] arrays")
    nv = np.ascontiguousarray((am != 0).sum(1), np.int32)
    if ((am != 0) != (np.arange(shape[1])[None, :] < nv[:, None])).any():
        raise ValueError("attention_mask must be a prefix mask (ones, then the zero padding)")
    return nv


class _Trainer(_Handle):
    """One pllb_train_* handle (encoder, AdamW, stateless dropout, CUDA graphs) and the state_dict keys it was
    created from.  A subclass creates the handle and names its encoder keys, head pointers and aliases."""

    _DESTROY = "pllb_train_destroy"
    _HEAD_KEYS = ()       # keys passed to the export calls as extra device pointers, after pllb_weights

    def __init__(self, state_dict, cfg, device, lr, hidden_dropout, attention_dropout, seed, max_rows, max_seq, betas, eps,
                 weight_decay, pad_id):
        import torch
        from .synth import config_from_state_dict

        self._lib = _lib.load()
        _lib.require_device()
        self._h = ctypes.c_void_p()
        self.cfg = dict(cfg) if cfg is not None else config_from_state_dict(state_dict)
        self.device = device
        self._dev = torch.device("cuda", device)
        self._keys = list(state_dict.keys())
        self._passthrough = {k: v for k, v in state_dict.items() if self._passes_through(k)}
        self._shapes = {k: tuple(v.shape) for k, v in state_dict.items()}
        self.max_seq = min(int(max_seq), int(self.cfg["max_position"]), 512)
        self._desc = _model_desc(self.cfg)
        self._train_desc = TrainDesc(float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                                     float(hidden_dropout), float(attention_dropout), int(seed) & (2 ** 64 - 1), int(pad_id),
                                     int(max_rows), self.max_seq)

    def _passes_through(self, key: str) -> bool:
        """Keys the trainer does not hold: export returns the given tensor."""
        return key.endswith("position_ids")

    def _encoder_keys(self):
        return self._keys

    def _alias(self, key: str) -> str:
        return key

    def _to_dev(self, t):
        import torch
        return t.detach().to(device=self._dev, dtype=torch.float32).contiguous()

    def _weights_in(self, state_dict):
        """pllb_weights over device fp32 copies of the encoder tensors, ready for the create call."""
        import torch
        w, keep = weights_struct(lambda key: self._to_dev(state_dict[key]), self.cfg["num_layers"], self._encoder_keys())
        torch.cuda.synchronize(self._dev)
        return w, keep

    def _export(self, fn) -> Dict[str, "torch.Tensor"]:
        """fn(handle, pllb_weights, *head pointers) fills one zeroed device tensor per key (aliased keys share one);
        returns CPU tensors under the keys given at construction."""
        import torch
        bufs = {}

        def get(key):
            key = self._alias(key)
            if key not in bufs:
                bufs[key] = torch.zeros(self._shapes[key], dtype=torch.float32, device=self._dev)
            return bufs[key]

        w, keep = weights_struct(get, self.cfg["num_layers"], self._encoder_keys())
        head = [ctypes.c_void_p(get(k).data_ptr()) for k in self._HEAD_KEYS]
        torch.cuda.synchronize(self._dev)
        check(fn(self._h, ctypes.byref(w), *head))
        torch.cuda.synchronize(self._dev)
        host = {k: v.cpu() for k, v in bufs.items()}
        del keep
        return {k: self._passthrough[k] if k in self._passthrough else host[self._alias(k)] for k in self._keys}

    def reset_optimizer(self, lr: float):
        """A fresh AdamW: zero moments, step count 0, learning rate lr (the reference creates one per epoch,
        MLM_PLL/main.py:76)."""
        check(self._lib.pllb_train_reset_optimizer(self._h, float(lr)))

    def workspace_bytes(self) -> int:
        return int(self._lib.pllb_train_workspace_bytes(self._h))

    def kernel_launches(self) -> int:
        return int(self._lib.pllb_train_kernel_launches(self._h))

    def graph_replays(self) -> int:
        """Steps that ran as replays of a captured CUDA graph (PLLB_TRAIN_GRAPH=0 disables capture)."""
        return int(self._lib.pllb_train_graph_replays(self._h))


class MlmTrainer(_Trainer):
    """BERT masked-LM fine-tuning on the device; stands in for ``BertForMaskedLM`` (train mode) +
    ``torch.optim.AdamW`` inside ``run_one_epoch(train_mode=True)`` (MLM_PLL/main.py:73-99) and for
    the loss-only dev pass (train_mode=False, do_scoring=False).  fp32 master weights, bf16 GEMM
    operands, fp32 accumulation.  ``hidden_dropout`` / ``attention_dropout`` default to the
    BertConfig values of bert-base-chinese (0.1); the masks come from a stateless hash of
    (seed, step, site, element), not from torch's RNG, so only runs with dropout 0 are comparable
    value by value with the reference."""

    TIED = {"cls.predictions.decoder.weight": "bert.embeddings.word_embeddings.weight",
            "cls.predictions.decoder.bias": "cls.predictions.bias"}

    def __init__(self, state_dict: Dict[str, "torch.Tensor"], cfg: Optional[dict] = None, device: int = 0,
                 lr: float = 1e-5, hidden_dropout: float = 0.1, attention_dropout: float = 0.1, seed: int = 0,
                 max_rows: int = 4096, max_seq: int = 128, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.01, pad_id: int = 0):
        super().__init__(state_dict, cfg, device, lr, hidden_dropout, attention_dropout, seed, max_rows, max_seq, betas, eps,
                         weight_decay, pad_id)
        if "cls.predictions.transform.dense.weight" not in state_dict:
            raise ValueError("MLM fine-tuning needs a BertForMaskedLM state_dict (cls.predictions.* missing)")
        w, keep = self._weights_in(state_dict)
        check(self._lib.pllb_train_create(ctypes.byref(self._h), ctypes.byref(self._desc), ctypes.byref(w),
                                          ctypes.byref(self._train_desc), device))
        del keep

    def _alias(self, key: str) -> str:
        """Tied entries are one tensor, as in model.state_dict()."""
        src = self.TIED.get(key, key)
        return src if src in self._shapes else key

    def step(self, input_ids, attention_mask, labels, mode: int = 1) -> float:
        """One zero-padded batch (int arrays [B, T], what collate builds).  mode 1: forward + backward
        + AdamW step; 0: loss only (eval); 2: forward + backward without the update.  Returns the loss."""
        ids = np.ascontiguousarray(input_ids, np.int32)
        lab = np.ascontiguousarray(labels, np.int32)
        if ids.ndim != 2 or lab.shape != ids.shape:
            raise ValueError("input_ids, attention_mask and labels must be equal [B, T] arrays")
        nv = _prefix_lengths(attention_mask, ids.shape)
        loss = ctypes.c_float(0.0)
        check(self._lib.pllb_train_step_host(self._h, _np_ptr(ids), _np_ptr(nv), _np_ptr(lab), ids.shape[0], ids.shape[1],
                                             int(mode), ctypes.byref(loss)))
        return float(loss.value)

    def row_losses(self, n_rows: int) -> np.ndarray:
        """-log_softmax(logits)[labels] of every position of the last step (float32 [B*T], row-major)."""
        out = np.zeros(int(n_rows), np.float32)
        check(self._lib.pllb_train_row_losses_host(self._h, _np_ptr(out), int(n_rows)))
        return out

    def state_dict(self) -> Dict[str, "torch.Tensor"]:
        """fp32 CPU tensors under the keys of the state_dict given at construction (model.state_dict(),
        MLM_PLL/main.py:155)."""
        return self._export(self._lib.pllb_train_export)

    def grads(self) -> Dict[str, "torch.Tensor"]:
        """Gradients of the last mode-1 / mode-2 step, same keys (parity tests)."""
        return self._export(self._lib.pllb_train_export_grads)


class ClsTrainer(_Trainer):
    """RescoreBert distillation on the device: the student of RescoreBert/model.py (BertModel, then
    Linear(H, 1) on the [CLS] state) trained with the MD loss (MSE to the teacher PLL) and, optionally,
    the MWER loss over each utterance's N-best list (include/pllb.h, pllb_cls_train_*, states the
    formulas).  Same encoder, optimizer (AdamW, weight decay on every parameter, linear.* included),
    stateless dropout and CUDA graphs as :class:`MlmTrainer`; only runs with dropout 0 are comparable
    value by value with an fp32 reference.

    ``state_dict``: ``bert.*`` (a BertModel, with or without ``bert.pooler.*``), ``linear.weight``
    [1, H], ``linear.bias`` [1].  The pooler is not used by the score and gets no gradient: it comes
    back from :meth:`state_dict` unchanged."""

    POOLER = "bert.pooler."
    _HEAD_KEYS = ("linear.weight", "linear.bias")

    def __init__(self, state_dict: Dict[str, "torch.Tensor"], cfg: Optional[dict] = None, device: int = 0,
                 lr: float = 1e-5, md_weight: float = 1.0, mwer_weight: float = 0.0, am_weight: float = 1.0,
                 hidden_dropout: float = 0.1, attention_dropout: float = 0.1, seed: int = 0, max_rows: int = 4096,
                 max_seq: int = 128, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.01, pad_id: int = 0):
        if "linear.weight" not in state_dict or "linear.bias" not in state_dict:
            raise ValueError("RescoreBert training needs linear.weight [1, H] and linear.bias [1] in the state_dict")
        super().__init__(state_dict, cfg, device, lr, hidden_dropout, attention_dropout, seed, max_rows, max_seq, betas, eps,
                         weight_decay, pad_id)
        if state_dict["linear.weight"].numel() != self.cfg["hidden"] or state_dict["linear.bias"].numel() != 1:
            raise ValueError("linear.weight must have `hidden` elements and linear.bias one")
        lw, lb = (self._to_dev(state_dict[k]).reshape(-1) for k in self._HEAD_KEYS)
        w, keep = self._weights_in(state_dict)
        self.loss_weights = dict(md_weight=float(md_weight), mwer_weight=float(mwer_weight), am_weight=float(am_weight))
        ld = ClsLossDesc(**self.loss_weights)
        check(self._lib.pllb_cls_train_create(ctypes.byref(self._h), ctypes.byref(self._desc), ctypes.byref(w),
                                              ctypes.c_void_p(lw.data_ptr()), ctypes.c_void_p(lb.data_ptr()),
                                              ctypes.byref(self._train_desc), ctypes.byref(ld), device))
        del keep, lw, lb

    def _passes_through(self, key: str) -> bool:
        return super()._passes_through(key) or key.startswith(self.POOLER)

    def _encoder_keys(self):
        return [k for k in self._keys if k.startswith("bert.") and not k.startswith(self.POOLER)]

    def step(self, input_ids, attention_mask, group, target, am, err, mode: int = 1):
        """One batch of whole utterances: input_ids / attention_mask int [B, T] ([CLS] t [SEP], zero-padded,
        prefix masks); group int [B] (0, 0, ..., 1, 1, ...: the utterance of each row); target (teacher PLL),
        am (AM score), err (CER) float [B].  mode 1: forward + backward + AdamW step; 0: loss only (eval);
        2: forward + backward without the update.  Returns (loss, float32 [B] scores of this forward pass)."""
        ids = np.ascontiguousarray(input_ids, np.int32)
        if ids.ndim != 2:
            raise ValueError("input_ids must be a [B, T] array")
        nv = _prefix_lengths(attention_mask, ids.shape)
        B = ids.shape[0]
        grp = np.ascontiguousarray(group, np.int32)
        vals = [np.ascontiguousarray(x, np.float32) for x in (target, am, err)]
        if grp.shape != (B,) or any(v.shape != (B,) for v in vals):
            raise ValueError("group, target, am and err must have one entry per row of input_ids")
        loss = ctypes.c_float(0.0)
        scores = np.zeros(B, np.float32)
        check(self._lib.pllb_cls_train_step_host(self._h, _np_ptr(ids), _np_ptr(nv), _np_ptr(grp), *map(_np_ptr, vals),
                                                 B, ids.shape[1], int(mode), ctypes.byref(loss), _np_ptr(scores)))
        return float(loss.value), scores

    def state_dict(self) -> Dict[str, "torch.Tensor"]:
        """fp32 CPU tensors under the keys of the state_dict given at construction; the pooler and
        position_ids entries are the given tensors.  ``RescoreBert(trainer.state_dict())`` scores with it."""
        return self._export(self._lib.pllb_cls_train_export)

    def grads(self) -> Dict[str, "torch.Tensor"]:
        """Gradients of the last mode-1 / mode-2 step under the same keys (zeros for the pooler;
        position_ids passes through)."""
        import torch
        g = self._export(self._lib.pllb_cls_train_export_grads)
        for k in g:
            if k.startswith(self.POOLER):
                g[k] = torch.zeros(self._shapes[k], dtype=torch.float32)      # the pooler gets no gradient
        return g


# ---------------------------------------------------------------------- stage 4
def pack_strings(strings: Sequence[str]):
    """Strings -> (code points int32[sum len], offsets int64[n+1]); len = Python code points."""
    off = np.zeros(len(strings) + 1, np.int64)
    if len(strings):
        np.cumsum(np.fromiter(map(len, strings), np.int64, len(strings)), out=off[1:])
    cp = np.frombuffer("".join(strings).encode("utf-32-le", "surrogatepass"), np.int32).copy()
    assert len(cp) == off[-1]
    return cp, off


_WS = None


def _whitespace_code_points() -> np.ndarray:
    """Code points str.strip() removes (str.isspace()), for the vectorised strip check."""
    global _WS
    if _WS is None:
        _WS = np.array([c for c in range(0x3001) if chr(c).isspace()], np.int32)   # none above U+3000
    return _WS


def pack_stripped(strings: Sequence[str]):
    """pack_strings([s.strip() for s in strings]) plus the RAW lengths, in one pass over the list:
    the strings are packed unstripped, and only if some string starts or ends with a whitespace
    code point (checked on the packed array) is the per-string strip() done.  Returns
    (code points, offsets, raw lengths int64)."""
    n = len(strings)
    raw_len = np.fromiter(map(len, strings), np.int64, n) if n else np.zeros(0, np.int64)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(raw_len, out=off[1:])
    cp = np.frombuffer("".join(strings).encode("utf-32-le", "surrogatepass"), np.int32)
    assert len(cp) == off[-1]
    nz = raw_len > 0
    ws = _whitespace_code_points()
    if nz.any() and (np.isin(cp[off[:-1][nz]], ws).any() or np.isin(cp[off[1:][nz] - 1], ws).any()):
        cp, off = pack_strings([s.strip() for s in strings])
        return cp, off, raw_len
    return cp.copy(), off, raw_len


def tokenize_packed(table: np.ndarray, cp: np.ndarray, cp_off: np.ndarray):
    """pllb_tokenize_host: packed code points -> (ids int32, offsets int64[n+1], needs_host uint8[n])."""
    lib = _lib.load()
    _lib.require_device()
    table = np.ascontiguousarray(table, np.int32)
    cp = np.ascontiguousarray(cp, np.int32)
    cp_off = np.ascontiguousarray(cp_off, np.int64)
    n = len(cp_off) - 1
    ids = np.zeros(max(int(cp_off[-1] - cp_off[0]), 1), np.int32)
    off = np.zeros(n + 1, np.int64)
    flag = np.zeros(max(n, 1), np.uint8)
    check(lib.pllb_tokenize_host(_np_ptr(table), len(table), _np_ptr(cp), _np_ptr(cp_off), n, _np_ptr(ids), _np_ptr(off),
                                 _np_ptr(flag)))
    return ids[:int(off[-1])], off, flag[:n]


def levenshtein_packed(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref) -> np.ndarray:
    """Edit distances of (ref[pair_ref[i]], hyp[i]) pairs on the GPU (host arrays in/out)."""
    lib = _lib.load()
    _lib.require_device()
    ref_cp = np.ascontiguousarray(ref_cp, np.int32)
    hyp_cp = np.ascontiguousarray(hyp_cp, np.int32)
    ref_off = np.ascontiguousarray(ref_off, np.int64)
    hyp_off = np.ascontiguousarray(hyp_off, np.int64)
    pair_ref = np.ascontiguousarray(pair_ref, np.int32)
    out = np.zeros(len(pair_ref), np.int32)
    check(lib.pllb_levenshtein_host(_np_ptr(ref_cp), _np_ptr(ref_off), len(ref_off) - 1, _np_ptr(hyp_cp),
                                    _np_ptr(hyp_off), _np_ptr(pair_ref), len(pair_ref), _np_ptr(out)))
    return out


def levenshtein(refs: Sequence[str], hyps: Sequence[str], pair_ref: Optional[Sequence[int]] = None) -> np.ndarray:
    """jiwer-style character edit distance: strings are stripped, characters = code points."""
    refs = [r.strip() for r in refs]
    hyps = [h.strip() for h in hyps]
    rc, ro = pack_strings(refs)
    hc, ho = pack_strings(hyps)
    if pair_ref is None:
        if len(refs) != len(hyps):
            raise ValueError("reference and hypothesis lists differ in length")
        pair_ref = np.arange(len(hyps), dtype=np.int32)
    return levenshtein_packed(rc, ro, hc, ho, pair_ref)


class Alignment:
    """Edit operations of n aligned pairs (DESIGN.md §3.10), as pllb_align_host returns them.

    ops: uint8 ASCII 'U'/'S'/'I'/'D'; pair i's ops are ops[off[i] : off[i] + n_ops[i]] (its slot
    runs to off[i+1] = off[i] + na + nb).  counts: int32 [n, 4] = (U, S, I, D) per pair."""

    LETTERS = "USID"

    def __init__(self, ops: np.ndarray, off: np.ndarray, n_ops: np.ndarray, counts: np.ndarray):
        self.ops, self.off, self.n_ops, self.counts = ops, off, n_ops, counts

    def __len__(self) -> int:
        return len(self.n_ops)

    def __getitem__(self, i: int) -> np.ndarray:
        o = int(self.off[i])
        return self.ops[o:o + int(self.n_ops[i])]

    def op_string(self, i: int) -> str:
        return self[i].tobytes().decode("ascii")


def align_packed(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref) -> Alignment:
    """Edit-operation alignment of (ref[pair_ref[i]], hyp i) pairs on the GPU (host arrays in/out).
    Symbols are opaque int32; one kernel launch for every pair."""
    lib = _lib.load()
    _lib.require_device()
    ref_cp = np.ascontiguousarray(ref_cp, np.int32)
    hyp_cp = np.ascontiguousarray(hyp_cp, np.int32)
    ref_off = np.ascontiguousarray(ref_off, np.int64)
    hyp_off = np.ascontiguousarray(hyp_off, np.int64)
    pair_ref = np.ascontiguousarray(pair_ref, np.int32)
    n = len(pair_ref)
    n_ref = len(ref_off) - 1
    # slot of pair i: na + nb bytes.  An out-of-range pair_ref gets a 0-length ref here; the
    # library rejects it before it reads the offsets.
    ok = (pair_ref >= 0) & (pair_ref < n_ref)
    na = np.diff(ref_off)[np.where(ok, pair_ref, 0)] if n_ref > 0 else np.zeros(n, np.int64)
    off = np.zeros(n + 1, np.int64)
    if n:
        np.cumsum(np.where(ok, na, 0) + np.diff(hyp_off), out=off[1:])
    ops = np.zeros(max(int(off[-1]), 1), np.uint8)
    n_ops = np.zeros(n, np.int32)
    counts = np.zeros((n, 4), np.int32)
    check(lib.pllb_align_host(_np_ptr(ref_cp), _np_ptr(ref_off), n_ref, _np_ptr(hyp_cp), _np_ptr(hyp_off),
                              _np_ptr(pair_ref), n, _np_ptr(off), _np_ptr(ops), _np_ptr(n_ops), _np_ptr(counts)))
    return Alignment(ops[:int(off[-1])], off, n_ops, counts)


def align(refs: Sequence[str], hyps: Sequence[str], pair_ref: Optional[Sequence[int]] = None) -> Alignment:
    """Character edit-operation alignment; strings are stripped like engine.levenshtein, so
    S + I + D of a pair equals its levenshtein distance."""
    refs = [r.strip() for r in refs]
    hyps = [h.strip() for h in hyps]
    rc, ro = pack_strings(refs)
    hc, ho = pack_strings(hyps)
    if pair_ref is None:
        if len(refs) != len(hyps):
            raise ValueError("reference and hypothesis lists differ in length")
        pair_ref = np.arange(len(hyps), dtype=np.int32)
    return align_packed(rc, ro, hc, ho, pair_ref)


def rescore_sweep(am, lm, lens, dist, weights, variant="B"):
    """For every weight: per-utterance argmax of the interpolated score and the summed edit
    distance of the chosen hypotheses.  Returns (argmax int32 [W,N], edit_sum int64 [W])."""
    lib = _lib.load()
    _lib.require_device()
    am = np.ascontiguousarray(am, np.float64)
    lm = np.ascontiguousarray(lm, np.float64)
    lens = np.ascontiguousarray(lens, np.int64)
    weights = np.ascontiguousarray(weights, np.float64)
    if am.shape != lm.shape or am.shape != lens.shape or am.ndim != 2:
        raise ValueError(f"am {am.shape}, lm {lm.shape}, len {lens.shape} must be equal 2-D shapes")
    N, nb = am.shape
    W = len(weights)
    arg = np.zeros((W, N), np.int32)
    es = np.zeros(W, np.int64)
    d = None
    if dist is not None:
        d = np.ascontiguousarray(dist, np.int32)
        if d.shape != am.shape:
            raise ValueError("dist shape mismatch")
    check(lib.pllb_rescore_sweep_host(_np_ptr(am), _np_ptr(lm), _np_ptr(lens), _np_ptr(d) if d is not None else None,
                                      N, nb, _np_ptr(weights), W, VARIANTS[variant], _np_ptr(arg), _np_ptr(es)))
    return arg, es


def rescore_scores(am, lm, lens, weight, variant="B") -> np.ndarray:
    """The [N, n_best] interpolated score matrix for one weight (rescore.py:47-53)."""
    import torch
    lib = _lib.load()
    _lib.require_device()
    am = np.ascontiguousarray(am, np.float64)
    lm = np.ascontiguousarray(lm, np.float64)
    lens = np.ascontiguousarray(lens, np.int64)
    if am.shape != lm.shape or am.shape != lens.shape or am.ndim != 2:
        raise ValueError(f"am {am.shape}, lm {lm.shape}, len {lens.shape} must be equal 2-D shapes")
    N, nb = am.shape
    dev = torch.device("cuda", torch.cuda.current_device())
    d_am, d_lm, d_len = (torch.from_numpy(x).to(dev) for x in (am, lm, lens))
    out = torch.empty(N, nb, dtype=torch.float64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    check(lib.pllb_rescore_scores(ctypes.c_void_p(d_am.data_ptr()), ctypes.c_void_p(d_lm.data_ptr()),
                                  ctypes.c_void_p(d_len.data_ptr()), N, nb, float(weight), VARIANTS[variant],
                                  ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(stream)))
    torch.cuda.synchronize(dev)
    return out.cpu().numpy()


def debug_gemm(A_bf16, W_bf16, bias_f32, epilogue: int, simt: bool = False, operand_dtype: str = "bf16"):
    """Test hook: C = A @ W^T + bias through the tcgen05 (or SIMT validation) kernel.
    operand_dtype "fp16": A and W are torch.float16."""
    import torch
    lib = _lib.load()
    _lib.require_device()
    M, K = A_bf16.shape
    N = W_bf16.shape[0]
    out = torch.empty(M, N, dtype=A_bf16.dtype if epilogue in (0, 1) else torch.float32, device=A_bf16.device)
    stream = torch.cuda.current_stream(A_bf16.device).cuda_stream
    args = (ctypes.c_void_p(A_bf16.data_ptr()), ctypes.c_void_p(W_bf16.data_ptr()), ctypes.c_void_p(bias_f32.data_ptr()),
            ctypes.c_void_p(out.data_ptr()), M, N, K, epilogue)
    if simt:
        check(lib.pllb_debug_gemm_simt(*args, ctypes.c_void_p(stream)))
    elif operand_dtype == "bf16":
        check(lib.pllb_debug_gemm(*args, ctypes.c_void_p(stream)))
    else:
        check(lib.pllb_debug_gemm_dt(*args, OPERAND_DTYPES[operand_dtype], ctypes.c_void_p(stream)))
    return out


# ---------------------------------------------------------------------------------------------- seq2seq
# BartForConditionalGeneration (CorrectBart, DESIGN.md §3.11): the HF state_dict names of every tensor the
# library takes, keyed by where it goes.  `cfg` is a BartConfig.to_dict()-style dict.
_BART_ENC_LAYER = {"q_w": "self_attn.q_proj.weight", "q_b": "self_attn.q_proj.bias",
                   "k_w": "self_attn.k_proj.weight", "k_b": "self_attn.k_proj.bias",
                   "v_w": "self_attn.v_proj.weight", "v_b": "self_attn.v_proj.bias",
                   "ao_w": "self_attn.out_proj.weight", "ao_b": "self_attn.out_proj.bias",
                   "ao_ln_g": "self_attn_layer_norm.weight", "ao_ln_b": "self_attn_layer_norm.bias",
                   "ff1_w": "fc1.weight", "ff1_b": "fc1.bias", "ff2_w": "fc2.weight", "ff2_b": "fc2.bias",
                   "out_ln_g": "final_layer_norm.weight", "out_ln_b": "final_layer_norm.bias"}
_BART_DEC_LAYER = {"q_w": "self_attn.q_proj.weight", "q_b": "self_attn.q_proj.bias",
                   "k_w": "self_attn.k_proj.weight", "k_b": "self_attn.k_proj.bias",
                   "v_w": "self_attn.v_proj.weight", "v_b": "self_attn.v_proj.bias",
                   "o_w": "self_attn.out_proj.weight", "o_b": "self_attn.out_proj.bias",
                   "self_ln_g": "self_attn_layer_norm.weight", "self_ln_b": "self_attn_layer_norm.bias",
                   "cq_w": "encoder_attn.q_proj.weight", "cq_b": "encoder_attn.q_proj.bias",
                   "ck_w": "encoder_attn.k_proj.weight", "ck_b": "encoder_attn.k_proj.bias",
                   "cv_w": "encoder_attn.v_proj.weight", "cv_b": "encoder_attn.v_proj.bias",
                   "co_w": "encoder_attn.out_proj.weight", "co_b": "encoder_attn.out_proj.bias",
                   "cross_ln_g": "encoder_attn_layer_norm.weight", "cross_ln_b": "encoder_attn_layer_norm.bias",
                   "ff1_w": "fc1.weight", "ff1_b": "fc1.bias", "ff2_w": "fc2.weight", "ff2_b": "fc2.bias",
                   "final_ln_g": "final_layer_norm.weight", "final_ln_b": "final_layer_norm.bias"}
_BART_TOP = {"shared": "model.shared.weight",
             "enc_pos": "model.encoder.embed_positions.weight",
             "enc_ln_g": "model.encoder.layernorm_embedding.weight", "enc_ln_b": "model.encoder.layernorm_embedding.bias",
             "dec_pos": "model.decoder.embed_positions.weight",
             "dec_ln_g": "model.decoder.layernorm_embedding.weight", "dec_ln_b": "model.decoder.layernorm_embedding.bias",
             "final_logits_bias": "final_logits_bias"}
# tied copies of model.shared.weight a checkpoint may carry
BART_TIED_KEYS = ("model.encoder.embed_tokens.weight", "model.decoder.embed_tokens.weight", "lm_head.weight")


def bart_weight_keys(cfg: dict) -> Dict[tuple, str]:
    """{("top", name) | ("enc", layer, field) | ("dec", layer, field): state_dict key}."""
    out = {("top", k): v for k, v in _BART_TOP.items()}
    for i in range(int(cfg["encoder_layers"])):
        for f, k in _BART_ENC_LAYER.items():
            out[("enc", i, f)] = f"model.encoder.layers.{i}.{k}"
    for i in range(int(cfg["decoder_layers"])):
        for f, k in _BART_DEC_LAYER.items():
            out[("dec", i, f)] = f"model.decoder.layers.{i}.{k}"
    return out


def bart_state_dict(state_dict) -> Dict[str, "torch.Tensor"]:
    """The state_dict with one leading module prefix (a wrapper's ``bart.``) stripped, located by
    ``model.shared.weight``; tied copies of the shared table must equal it (ValueError otherwise)."""
    import torch
    anchor = [k for k in state_dict if k == "model.shared.weight" or k.endswith(".model.shared.weight")]
    if len(anchor) != 1:
        raise ValueError("state_dict must hold exactly one 'model.shared.weight' (optionally under one prefix)")
    prefix = anchor[0][:-len("model.shared.weight")]
    sd = {k[len(prefix):]: v for k, v in state_dict.items() if k.startswith(prefix)}
    shared = sd["model.shared.weight"]
    for k in BART_TIED_KEYS:
        if k in sd and not torch.equal(sd[k].detach().cpu(), shared.detach().cpu()):
            raise ValueError(f"{k} is not a copy of model.shared.weight: untied embeddings are not supported")
    return sd


def check_bart_config(cfg: dict) -> dict:
    """The library's s2s shape from a BartConfig dict; ValueError for what the kernels do not implement."""
    H = int(cfg["d_model"])
    heads = int(cfg["encoder_attention_heads"])
    if cfg.get("activation_function", "gelu") != "gelu":
        raise ValueError("only activation_function 'gelu' (erf form) is supported")
    if cfg.get("normalize_before", False) or cfg.get("add_final_layer_norm", False):
        raise ValueError("only post-LN BART (no normalize_before / final layer_norm) is supported")
    if int(cfg.get("decoder_attention_heads", heads)) != heads or heads * 64 != H:
        raise ValueError("head dim must be 64 in both stacks")
    if H % 256 or not 256 <= H <= 1024 or int(cfg["encoder_ffn_dim"]) % 256 or int(cfg["decoder_ffn_dim"]) % 256:
        raise ValueError("d_model must be 256/512/768/1024 and the FFN widths multiples of 256")
    return dict(enc_layers=int(cfg["encoder_layers"]), dec_layers=int(cfg["decoder_layers"]), hidden=H, num_heads=heads,
                enc_intermediate=int(cfg["encoder_ffn_dim"]), dec_intermediate=int(cfg["decoder_ffn_dim"]),
                vocab=int(cfg["vocab_size"]), max_position=int(cfg["max_position_embeddings"]),
                embed_scale=float(np.sqrt(H)) if cfg.get("scale_embedding", False) else 1.0)


def s2s_weights_struct(get, cfg: dict, pos_skip_rows: int):
    """pllb_s2s_weights over the device fp32 tensors ``get(key)`` returns for the BART state_dict names; the two
    position tables start ``pos_skip_rows`` rows in (2 for pllb_s2s_create, 0 for pllb_s2s_train_create).  Returns
    (struct, list keeping the tensors and the layer arrays alive)."""
    from ._lib import DecLayerWeights, S2sWeights
    s = check_bart_config(cfg)
    keep = []

    def dp(key, skip_rows: int = 0):
        t = get(key)[skip_rows:].contiguous()
        keep.append(t)
        return ctypes.c_void_p(t.data_ptr())

    enc_layers = (LayerWeights * s["enc_layers"])()
    dec_layers = (DecLayerWeights * s["dec_layers"])()
    keep += [enc_layers, dec_layers]
    for (kind, *rest), key in bart_weight_keys(cfg).items():
        if kind == "enc":
            setattr(enc_layers[rest[0]], rest[1], dp(key))
        elif kind == "dec":
            setattr(dec_layers[rest[0]], rest[1], dp(key))
    w = S2sWeights()
    w.enc.pos_emb = dp(_BART_TOP["enc_pos"], pos_skip_rows)
    w.enc.emb_ln_g, w.enc.emb_ln_b = dp(_BART_TOP["enc_ln_g"]), dp(_BART_TOP["enc_ln_b"])
    w.enc.layers = ctypes.cast(enc_layers, ctypes.POINTER(LayerWeights))
    w.dec_layers = ctypes.cast(dec_layers, ctypes.POINTER(DecLayerWeights))
    w.shared = dp(_BART_TOP["shared"])
    w.dec_pos_emb = dp(_BART_TOP["dec_pos"], pos_skip_rows)
    w.dec_emb_ln_g, w.dec_emb_ln_b = dp(_BART_TOP["dec_ln_g"]), dp(_BART_TOP["dec_ln_b"])
    w.final_logits_bias = dp("final_logits_bias")                     # [1, vocab] or [vocab]
    return w, keep


_GEN_KEYS = ("max_length", "decoder_start_token_id", "eos_token_id", "pad_token_id", "forced_bos_token_id",
             "forced_eos_token_id")


def generation_settings(cfg: dict, **overrides) -> dict:
    """generate()'s settings from a config dict (+ overrides), checked as pllb_generate checks them:
    ValueError for beam search, sampling, no_repeat_ngram_size, min_length, repetition_penalty != 1 and
    ids outside the vocabulary."""
    g = {k: cfg.get(k) for k in _GEN_KEYS}
    for k in ("num_beams", "do_sample", "no_repeat_ngram_size", "min_length", "repetition_penalty"):
        if k in cfg:
            g[k] = cfg[k]
    g.update(overrides)
    if g.get("max_length") is None:
        g["max_length"] = 20
    if int(g.get("num_beams") or 1) != 1:
        raise ValueError("beam search (num_beams > 1) is not supported; greedy only")
    if g.get("do_sample"):
        raise ValueError("sampling is not supported; greedy only")
    if int(g.get("no_repeat_ngram_size") or 0) != 0:
        raise ValueError("no_repeat_ngram_size is not supported")
    if int(g.get("min_length") or 0) != 0:
        raise ValueError("min_length is not supported")
    if float(g.get("repetition_penalty") if g.get("repetition_penalty") is not None else 1.0) != 1.0:
        raise ValueError("repetition_penalty != 1 is not supported")
    V = int(cfg["vocab_size"])
    ml = int(g["max_length"])
    if not 2 <= ml <= int(cfg["max_position_embeddings"]):
        raise ValueError(f"max_length must lie in [2, {cfg['max_position_embeddings']}]")
    for k in ("decoder_start_token_id", "eos_token_id", "pad_token_id"):
        if g[k] is None or not 0 <= int(g[k]) < V:
            raise ValueError(f"{k} must be an id inside the vocabulary")
    for k in ("forced_bos_token_id", "forced_eos_token_id"):
        if g[k] is not None and not 0 <= int(g[k]) < V:
            raise ValueError(f"{k} must be None or an id inside the vocabulary")
    return g


_EARLY_STOPPING = {False: 0, True: 1, "never": 2}


def beam_settings(cfg: dict, **overrides) -> dict:
    """generate()'s beam-search settings from a config dict (+ overrides), checked as pllb_generate_beam
    checks them: num_beams in [2, 8] with vocab >= 2 * num_beams, num_return_sequences in [1, num_beams]
    (default 1), a finite length_penalty (default 1.0) and early_stopping False / True / "never" (default
    False); everything else as generation_settings checks it.  ValueError otherwise."""
    g = {k: cfg.get(k) for k in _GEN_KEYS}
    for k in ("do_sample", "no_repeat_ngram_size", "min_length", "repetition_penalty"):
        if k in cfg:
            g[k] = cfg[k]
    for k, default in (("num_beams", None), ("num_return_sequences", 1), ("length_penalty", 1.0),
                       ("early_stopping", False)):
        g[k] = cfg.get(k, default) if cfg.get(k) is not None else default
    g.update(overrides)
    K = int(g.get("num_beams") or 1)
    if not 2 <= K <= 8:
        raise ValueError("num_beams must lie in [2, 8] for beam search")
    if int(cfg["vocab_size"]) < 2 * K:
        raise ValueError("beam search needs vocab_size >= 2 * num_beams")
    r = int(g["num_return_sequences"] if g["num_return_sequences"] is not None else 1)
    if not 1 <= r <= K:
        raise ValueError("num_return_sequences must lie in [1, num_beams]")
    lp = float(g["length_penalty"] if g["length_penalty"] is not None else 1.0)
    if not np.isfinite(lp):
        raise ValueError("length_penalty must be finite")
    es = g["early_stopping"]
    if not any(es is k or (isinstance(es, str) and es == k) for k in _EARLY_STOPPING):
        raise ValueError('early_stopping must be False, True or "never"')
    if K * int(g.get("max_length") or 20) > 12288:
        raise ValueError("num_beams * max_length must not exceed 12288")
    rest = generation_settings(cfg, **{k: v for k, v in g.items()
                                       if k not in ("num_beams", "num_return_sequences", "length_penalty",
                                                    "early_stopping")}, num_beams=1)
    rest.update(num_beams=K, num_return_sequences=r, length_penalty=lp, early_stopping=es)
    return rest


def _beam_desc(g: dict) -> "_lib.BeamDesc":
    es = g["early_stopping"]
    code = 2 if isinstance(es, str) else int(bool(es))
    return _lib.BeamDesc(int(g["num_return_sequences"]), float(g["length_penalty"]), code)


def _gen_desc(g: dict) -> "_lib.GenDesc":
    rp = g.get("repetition_penalty")
    return _lib.GenDesc(int(g["max_length"]), int(g["decoder_start_token_id"]), int(g["eos_token_id"]),
                        int(g["pad_token_id"]), -1 if g.get("forced_bos_token_id") is None else int(g["forced_bos_token_id"]),
                        -1 if g.get("forced_eos_token_id") is None else int(g["forced_eos_token_id"]),
                        int(g.get("num_beams") or 1), int(bool(g.get("do_sample"))), int(g.get("no_repeat_ngram_size") or 0),
                        int(g.get("min_length") or 0), float(1.0 if rp is None else rp))


class Seq2SeqGenerator(_Handle):
    """Greedy generation with a BartForConditionalGeneration state_dict (pllb_s2s_* / pllb_generate):
    the encoder reads [CLS] t [SEP], the decoder emits ids as ``generate(num_beams=1, do_sample=False)``."""

    _DESTROY = "pllb_s2s_destroy"

    def __init__(self, state_dict: Dict[str, "torch.Tensor"], cfg: dict, device: int = 0, max_rows: int = 0,
                 operand_dtype: str = "bf16", cls_id: int = 101, sep_id: int = 102):
        import torch
        from ._lib import S2sDesc

        self._lib = _lib.load()
        _lib.require_device()
        self._h = ctypes.c_void_p()
        self.cfg = dict(cfg)
        self.shape = check_bart_config(self.cfg)
        if operand_dtype not in ("bf16", "fp16"):
            raise ValueError("operand_dtype must be 'bf16' or 'fp16'")
        self.operand_dtype = operand_dtype
        sd = bart_state_dict(state_dict)
        dev = torch.device("cuda", device)
        s = self.shape
        H = s["hidden"]

        def get(key):
            if key not in sd:                                         # final_logits_bias: a missing buffer loads as zeros
                return torch.zeros(s["vocab"], dtype=torch.float32, device=dev)
            return sd[key].detach().to(device=dev, dtype=torch.float32)

        w, keep = s2s_weights_struct(get, self.cfg, pos_skip_rows=2)  # BartLearnedPositionalEmbedding's offset of 2
        d = S2sDesc(s["enc_layers"], s["dec_layers"], H, s["num_heads"], s["enc_intermediate"], s["dec_intermediate"],
                    s["vocab"], s["max_position"], s["max_position"],
                    1e-5, s["embed_scale"], cls_id, sep_id, 0 if operand_dtype == "bf16" else 1)
        torch.cuda.synchronize(dev)
        check(self._lib.pllb_s2s_create(ctypes.byref(self._h), ctypes.byref(d), ctypes.byref(w), int(max_rows), device))
        del keep

    def generate_packed(self, tokens: np.ndarray, offsets: np.ndarray, generation: dict, return_logits: bool = False):
        """HOST arrays in and out.  tokens int32 (no specials), offsets int64[n+1].  Returns
        (ids int32[n, max_length], lengths int32[n]) and with return_logits the fp32 logit of every chosen
        token (float32[n, max_length], 0 at position 0 and at pads)."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        tokens = np.ascontiguousarray(tokens, np.int32)
        if offsets.ndim != 1 or len(offsets) < 1:
            raise ValueError("offsets must be a 1-D array of n+1 entries")
        n = len(offsets) - 1
        ml = int(generation["max_length"])
        ids = np.zeros((n, ml), np.int32)
        lens = np.zeros(n, np.int32)
        lg = np.zeros((n, ml), np.float32) if return_logits else None
        g = _gen_desc(generation)
        check(self._lib.pllb_generate_host(self._h, ctypes.byref(g), _np_ptr(tokens) if len(tokens) else None,
                                           _np_ptr(offsets), n, _np_ptr(ids), _np_ptr(lens),
                                           _np_ptr(lg) if lg is not None else None))
        return (ids, lens, lg) if return_logits else (ids, lens)

    def beam_search_packed(self, tokens: np.ndarray, offsets: np.ndarray, settings: dict):
        """Beam search (pllb_generate_beam_host) with ``beam_settings``.  HOST arrays in and out; returns
        (ids int32[n, r, max_length], lengths int32[n, r], scores float32[n, r]), r = num_return_sequences,
        hypotheses in descending score order."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        tokens = np.ascontiguousarray(tokens, np.int32)
        if offsets.ndim != 1 or len(offsets) < 1:
            raise ValueError("offsets must be a 1-D array of n+1 entries")
        n, ml, r = len(offsets) - 1, int(settings["max_length"]), int(settings["num_return_sequences"])
        ids = np.zeros((n, r, ml), np.int32)
        lens = np.zeros((n, r), np.int32)
        scores = np.zeros((n, r), np.float32)
        g, b = _gen_desc(settings), _beam_desc(settings)
        check(self._lib.pllb_generate_beam_host(self._h, ctypes.byref(g), ctypes.byref(b),
                                                _np_ptr(tokens) if len(tokens) else None, _np_ptr(offsets), n,
                                                _np_ptr(ids), _np_ptr(lens), _np_ptr(scores)))
        return ids, lens, scores

    def debug_beam_replay(self, hidden: np.ndarray, settings: dict):
        """Test hook (pllb_s2s_debug_beam_replay): the LM head and beam selection alone on given decoder
        outputs hidden float32[max_length - 1, n * num_beams, d_model].  Returns (ids, lengths, scores) as
        beam_search_packed plus parents int32[steps, n * K] and running scores float32[steps, n * K]."""
        hidden = np.ascontiguousarray(hidden, np.float32)
        steps, rows, _ = hidden.shape
        K, ml, r = int(settings["num_beams"]), int(settings["max_length"]), int(settings["num_return_sequences"])
        n = rows // K
        ids = np.zeros((n, r, ml), np.int32)
        lens = np.zeros((n, r), np.int32)
        scores = np.zeros((n, r), np.float32)
        par = np.zeros((steps, rows), np.int32)
        rs = np.zeros((steps, rows), np.float32)
        g, b = _gen_desc(settings), _beam_desc(settings)
        check(self._lib.pllb_s2s_debug_beam_replay(self._h, ctypes.byref(g), ctypes.byref(b), n, _np_ptr(hidden), steps,
                                                   _np_ptr(ids), _np_ptr(lens), _np_ptr(scores), _np_ptr(par),
                                                   _np_ptr(rs)))
        return ids, lens, scores, par, rs

    def set_timing(self, enable: bool):
        check(self._lib.pllb_s2s_set_timing(self._h, int(enable)))

    def reset_stats(self):
        check(self._lib.pllb_s2s_reset_stats(self._h))

    def stats(self) -> dict:
        s = _lib.S2sStats()
        check(self._lib.pllb_s2s_get_stats(self._h, ctypes.byref(s)))
        d = {n: getattr(s, n) for n, _ in _lib.S2sStats._fields_}
        d["workspace_bytes"] = int(self._lib.pllb_s2s_workspace_bytes(self._h))
        return d


def shift_tokens_right(labels, pad_id: int, decoder_start_id: int) -> np.ndarray:
    """The decoder input pllb_s2s_train_step_host builds from labels [B, T_dec] (transformers'
    ``shift_tokens_right``): the start id at position 0, the labels shifted right by one, -100 -> pad_id."""
    lab = np.asarray(labels)
    out = np.empty(lab.shape, np.int64)
    out[:, 0] = decoder_start_id
    out[:, 1:] = lab[:, :-1]
    out[out == -100] = pad_id
    return out


class Seq2SeqTrainer(_Trainer):
    """CorrectBart fine-tuning on the device (pllb_s2s_train_*; include/pllb.h and DESIGN.md §3.13 state the
    contract): ``BartForConditionalGeneration.forward(input_ids, attention_mask, labels=labels)`` in train mode,
    ``loss.backward()`` and ``torch.optim.AdamW`` over ``model.parameters()``.  fp32 master weights, bf16 GEMM
    operands, fp32 accumulation.  ``dropout`` / ``attention_dropout`` default to the config's; the masks come from
    a stateless hash, so only runs with dropout 0 are comparable value by value with torch.

    ``state_dict``: a BartForConditionalGeneration state_dict (one wrapper prefix allowed, as
    :class:`Seq2SeqGenerator` takes it); ``cfg`` its BartConfig dict.  ``max_batch`` / ``max_enc_len`` /
    ``max_dec_len`` bound the batches :meth:`step` takes."""

    def __init__(self, state_dict: Dict[str, "torch.Tensor"], cfg: dict, device: int = 0, lr: float = 1e-5,
                 dropout: Optional[float] = None, attention_dropout: Optional[float] = None, seed: int = 0,
                 max_batch: int = 64, max_enc_len: int = 128, max_dec_len: int = 128, betas=(0.9, 0.999),
                 eps: float = 1e-8, weight_decay: float = 0.01, operand_dtype: str = "bf16"):
        import torch
        from ._lib import S2sDesc, S2sTrainDesc

        self.cfg = dict(cfg)
        self.shape = check_bart_config(self.cfg)
        if float(self.cfg.get("activation_dropout") or 0.0) != 0.0:
            raise ValueError("activation_dropout != 0 is not supported (bart-base's default is 0)")
        if operand_dtype != "bf16":
            raise ValueError("training takes bf16 GEMM operands only (no fp16 training)")
        sd = bart_state_dict(state_dict)
        # the handle is created here, not by _Trainer.__init__ (which builds the BERT descriptors)
        self._lib = _lib.load()
        _lib.require_device()
        self._h = ctypes.c_void_p()
        self.device = device
        self._dev = torch.device("cuda", device)
        self._keys = list(state_dict.keys())
        # bart_state_dict located exactly one model.shared.weight; its prefix maps the given keys to sd's
        self._prefix = next(k for k in state_dict if k == "model.shared.weight" or k.endswith(".model.shared.weight"))[
            :-len("model.shared.weight")]
        self._given = {k: v for k, v in state_dict.items()}
        self._shapes = {k: tuple(v.shape) for k, v in sd.items()}
        self.pad_id = int(self.cfg.get("pad_token_id", 0) if self.cfg.get("pad_token_id") is not None else 0)
        self.decoder_start_id = int(self.cfg["decoder_start_token_id"])
        s = self.shape
        if "final_logits_bias" not in sd:                              # a missing buffer loads as zeros in HF
            sd["final_logits_bias"] = torch.zeros(1, s["vocab"])
            self._shapes["final_logits_bias"] = (1, s["vocab"])
        w, keep = s2s_weights_struct(lambda k: self._to_dev(sd[k]), self.cfg, pos_skip_rows=0)
        self._desc = S2sDesc(s["enc_layers"], s["dec_layers"], s["hidden"], s["num_heads"], s["enc_intermediate"],
                             s["dec_intermediate"], s["vocab"], s["max_position"], s["max_position"], 1e-5,
                             s["embed_scale"], 101, 102, 0)
        drop = float(self.cfg.get("dropout", 0.1) if dropout is None else dropout)
        adrop = float(self.cfg.get("attention_dropout", 0.0) if attention_dropout is None else attention_dropout)
        self.max_batch, self.max_enc_len, self.max_dec_len = int(max_batch), int(max_enc_len), int(max_dec_len)
        self._train_desc = S2sTrainDesc(float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), drop,
                                        adrop, int(seed) & (2 ** 64 - 1), self.pad_id, self.decoder_start_id,
                                        self.max_batch, self.max_enc_len, self.max_dec_len)
        torch.cuda.synchronize(self._dev)
        check(self._lib.pllb_s2s_train_create(ctypes.byref(self._h), ctypes.byref(self._desc), ctypes.byref(w),
                                              ctypes.byref(self._train_desc), device))
        del keep
        self._last_shape = None

    def step(self, input_ids, attention_mask, labels, mode: int = 1) -> float:
        """One batch: input_ids / attention_mask int [B, T_enc] ([CLS] hyp [SEP], right-padded, prefix masks),
        labels int [B, T_dec] (-100 = ignored).  mode 1: forward + backward + AdamW step; 0: loss only (eval);
        2: forward + backward without the update.  Returns the loss."""
        ids = np.ascontiguousarray(input_ids, np.int32)
        lab = np.ascontiguousarray(labels, np.int32)
        if ids.ndim != 2 or lab.ndim != 2 or lab.shape[0] != ids.shape[0]:
            raise ValueError("input_ids [B, T_enc] and labels [B, T_dec] must be 2-D with the same B")
        nv = _prefix_lengths(attention_mask, ids.shape)
        loss = ctypes.c_float(0.0)
        check(self._lib.pllb_s2s_train_step_host(self._h, _np_ptr(ids), _np_ptr(nv), _np_ptr(lab), ids.shape[0],
                                                 ids.shape[1], lab.shape[1], int(mode), ctypes.byref(loss)))
        self._last_shape = lab.shape
        return float(loss.value)

    def token_losses(self) -> np.ndarray:
        """float32 [B, T_dec]: -log_softmax(logits)[label] of every decoder position of the last step, 0 where the
        label is -100."""
        if self._last_shape is None:
            raise RuntimeError("no step has run")
        out = np.zeros(self._last_shape, np.float32)
        check(self._lib.pllb_train_row_losses_host(self._h, _np_ptr(out), out.size))
        return out

    def _export(self, fn) -> Dict[str, "torch.Tensor"]:
        import torch
        bufs = {}

        def get(key):
            if key not in bufs:
                bufs[key] = torch.zeros(self._shapes[key], dtype=torch.float32, device=self._dev)
            return bufs[key]

        w, keep = s2s_weights_struct(get, self.cfg, pos_skip_rows=0)
        torch.cuda.synchronize(self._dev)
        check(fn(self._h, ctypes.byref(w)))
        torch.cuda.synchronize(self._dev)
        host = {k: v.cpu() for k, v in bufs.items()}
        del keep
        out = {}
        for k in self._keys:
            name = k[len(self._prefix):] if k.startswith(self._prefix) else k
            if name in BART_TIED_KEYS:
                name = _BART_TOP["shared"]
            out[k] = host[name].reshape(self._given[k].shape) if name in host else self._given[k]
        return out

    def state_dict(self) -> Dict[str, "torch.Tensor"]:
        """fp32 CPU tensors under the keys given at construction: the tied aliases hold the ``model.shared``
        values and ``final_logits_bias`` (a buffer) passes through.  ``CorrectBart(trainer.state_dict(), cfg,
        tokenizer)`` decodes with it."""
        return self._export(self._lib.pllb_s2s_train_export)

    def grads(self) -> Dict[str, "torch.Tensor"]:
        """Gradients of the last mode-1 / mode-2 step under the same keys (the tied aliases hold the one
        ``model.shared`` gradient; zeros for ``final_logits_bias``)."""
        import torch
        g = self._export(self._lib.pllb_s2s_train_export_grads)
        for k in g:
            if k.endswith("final_logits_bias"):
                g[k] = torch.zeros(self._given[k].shape, dtype=torch.float32)
        return g
