"""ctypes binding of libpllb200.so (include/pllb.h).  No fallback: if the library is
missing it is built with nvcc; if that fails, or no B200 is visible when a compute
entry point is called, an exception is raised."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_uint16, c_uint32, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PLLB_LIB") or os.path.join(HERE, "libpllb200.so")   # PLLB_LIB: A/B testing of builds


class PllbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libpllb200 error {code}: {msg}")
        self.code = code


class ModelDesc(ctypes.Structure):
    _fields_ = [("num_layers", c_int32), ("hidden", c_int32), ("num_heads", c_int32), ("intermediate", c_int32),
                ("vocab", c_int32), ("max_position", c_int32), ("ln_eps", c_float),
                ("cls_id", c_int32), ("sep_id", c_int32), ("mask_id", c_int32), ("operand_dtype", c_int32)]


_LAYER_FIELDS = ["q_w", "q_b", "k_w", "k_b", "v_w", "v_b", "ao_w", "ao_b", "ao_ln_g", "ao_ln_b",
                 "ff1_w", "ff1_b", "ff2_w", "ff2_b", "out_ln_g", "out_ln_b"]


class LayerWeights(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in _LAYER_FIELDS]


class Weights(ctypes.Structure):
    _fields_ = [("word_emb", c_void_p), ("pos_emb", c_void_p), ("type_emb", c_void_p), ("emb_ln_g", c_void_p),
                ("emb_ln_b", c_void_p), ("layers", POINTER(LayerWeights)), ("head_w", c_void_p), ("head_b", c_void_p),
                ("head_ln_g", c_void_p), ("head_ln_b", c_void_p), ("decoder_w", c_void_p), ("decoder_b", c_void_p)]


class Stats(ctypes.Structure):
    _fields_ = [("kernel_launches", c_int64), ("hyps_scored", c_int64), ("copies_scored", c_int64),
                ("tokens_expanded", c_int64), ("chunks", c_int64), ("gemm_flops", c_double),
                ("last_gemm_ms", c_float), ("last_total_ms", c_float), ("last_gemm_launches", c_int64)]


class TrainDesc(ctypes.Structure):
    _fields_ = [("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("adam_eps", c_float), ("weight_decay", c_float),
                ("hidden_dropout", c_float), ("attention_dropout", c_float), ("seed", c_uint64), ("pad_id", c_int32),
                ("max_rows", c_int32), ("max_seq", c_int32)]


class ClsLossDesc(ctypes.Structure):
    _fields_ = [("md_weight", c_float), ("mwer_weight", c_float), ("am_weight", c_float)]


class S2sDesc(ctypes.Structure):
    _fields_ = [("enc_layers", c_int32), ("dec_layers", c_int32), ("hidden", c_int32), ("num_heads", c_int32),
                ("enc_intermediate", c_int32), ("dec_intermediate", c_int32), ("vocab", c_int32),
                ("enc_max_position", c_int32), ("dec_max_position", c_int32), ("ln_eps", c_float),
                ("embed_scale", c_float), ("cls_id", c_int32), ("sep_id", c_int32), ("operand_dtype", c_int32)]


DEC_LAYER_FIELDS = ["q_w", "q_b", "k_w", "k_b", "v_w", "v_b", "o_w", "o_b", "self_ln_g", "self_ln_b",
                    "cq_w", "cq_b", "ck_w", "ck_b", "cv_w", "cv_b", "co_w", "co_b", "cross_ln_g", "cross_ln_b",
                    "ff1_w", "ff1_b", "ff2_w", "ff2_b", "final_ln_g", "final_ln_b"]


class DecLayerWeights(ctypes.Structure):
    _fields_ = [(n, c_void_p) for n in DEC_LAYER_FIELDS]


class S2sWeights(ctypes.Structure):
    _fields_ = [("enc", Weights), ("dec_layers", POINTER(DecLayerWeights)), ("shared", c_void_p),
                ("dec_pos_emb", c_void_p), ("dec_emb_ln_g", c_void_p), ("dec_emb_ln_b", c_void_p),
                ("final_logits_bias", c_void_p)]


class S2sTrainDesc(ctypes.Structure):
    _fields_ = [("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("adam_eps", c_float), ("weight_decay", c_float),
                ("dropout", c_float), ("attention_dropout", c_float), ("seed", c_uint64), ("pad_id", c_int32),
                ("decoder_start_id", c_int32), ("max_batch", c_int32), ("max_enc_len", c_int32), ("max_dec_len", c_int32)]


class GenDesc(ctypes.Structure):
    _fields_ = [("max_length", c_int32), ("decoder_start_id", c_int32), ("eos_id", c_int32), ("pad_id", c_int32),
                ("forced_bos_id", c_int32), ("forced_eos_id", c_int32), ("num_beams", c_int32), ("do_sample", c_int32),
                ("no_repeat_ngram_size", c_int32), ("min_length", c_int32), ("repetition_penalty", c_float)]


class BeamDesc(ctypes.Structure):
    _fields_ = [("num_return_sequences", c_int32), ("length_penalty", c_float), ("early_stopping", c_int32)]


class S2sStats(ctypes.Structure):
    _fields_ = [("kernel_launches", c_int64), ("steps", c_int64), ("chunks", c_int64), ("sentences", c_int64),
                ("gemm_flops", c_double), ("enc_ms", c_float), ("cross_kv_ms", c_float), ("dec_layers_ms", c_float),
                ("head_ms", c_float), ("total_ms", c_float)]


# name -> (restype, argtypes); every symbol include/pllb.h declares
SIGNATURES = {
    "pllb_last_error": (c_char_p, []),
    "pllb_abi_version": (c_int, []),
    "pllb_device_count": (c_int, []),
    "pllb_create": (c_int, [POINTER(c_void_p), POINTER(ModelDesc), POINTER(Weights), c_int64, c_int]),
    "pllb_destroy": (c_int, [c_void_p]),
    "pllb_workspace_bytes": (c_int64, [c_void_p]),
    "pllb_score": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "pllb_score_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "pllb_score_cls": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_float, c_void_p, c_void_p]),
    "pllb_score_cls_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_float, c_void_p]),
    "pllb_expand": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_get_stats": (c_int, [c_void_p, POINTER(Stats)]),
    "pllb_reset_stats": (c_int, [c_void_p]),
    "pllb_set_timing": (c_int, [c_void_p, c_int]),
    "pllb_get_gemm_breakdown": (c_int, [c_void_p, POINTER(c_float), POINTER(c_double)]),
    "pllb_debug_gemm": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "pllb_debug_gemm_dt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                   c_void_p]),
    "pllb_debug_gemm_simt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "pllb_debug_hidden": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "pllb_debug_train_attn": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_float, c_uint32,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_debug_s2s_attn": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32, c_int32,
                                    c_int32, c_int32, c_void_p, c_void_p, c_float, c_uint32, c_void_p, c_void_p, c_void_p,
                                    c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "pllb_debug_train_ln_fwd": (c_int, [c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_int32, c_void_p,
                                        c_void_p, c_float, c_void_p, c_void_p, c_float, c_int32, c_int32, c_void_p, c_float,
                                        c_uint32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_debug_train_ln_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p,
                                        c_float, c_int32, c_int32, c_void_p, c_void_p, c_void_p]),
    "pllb_debug_train_ce": (c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                    c_void_p]),
    "pllb_debug_train_embed_bwd": (c_int, [c_int32, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                           c_float, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_debug_train_colsum": (c_int, [c_void_p, c_int32, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                        c_void_p]),
    "pllb_debug_train_cast_transpose": (c_int, [c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                                                c_void_p]),
    "pllb_debug_train_gelu": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_embed": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "pllb_bertscore": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "pllb_tokenize_host": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "pllb_levenshtein": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p]),
    "pllb_levenshtein_host": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "pllb_align": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p,
                           c_void_p, c_void_p, c_void_p]),
    "pllb_align_host": (c_int, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "pllb_rescore_sweep": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32, c_int32,
                                   c_void_p, c_void_p, c_void_p]),
    "pllb_rescore_sweep_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_int32,
                                        c_int32, c_void_p, c_void_p]),
    "pllb_rescore_scores": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_double, c_int32, c_void_p, c_void_p]),
    "pllb_train_create": (c_int, [POINTER(c_void_p), POINTER(ModelDesc), POINTER(Weights), POINTER(TrainDesc), c_int]),
    "pllb_train_destroy": (c_int, [c_void_p]),
    "pllb_train_workspace_bytes": (c_int64, [c_void_p]),
    "pllb_train_kernel_launches": (c_int64, [c_void_p]),
    "pllb_train_graph_replays": (c_int64, [c_void_p]),
    "pllb_train_reset_optimizer": (c_int, [c_void_p, c_float]),
    "pllb_train_step_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, POINTER(c_float)]),
    "pllb_train_row_losses_host": (c_int, [c_void_p, c_void_p, c_int32]),
    "pllb_train_export": (c_int, [c_void_p, POINTER(Weights)]),
    "pllb_train_export_grads": (c_int, [c_void_p, POINTER(Weights)]),
    "pllb_cls_train_create": (c_int, [POINTER(c_void_p), POINTER(ModelDesc), POINTER(Weights), c_void_p, c_void_p,
                                      POINTER(TrainDesc), POINTER(ClsLossDesc), c_int]),
    "pllb_cls_train_step_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32,
                                         c_int32, c_int32, POINTER(c_float), c_void_p]),
    "pllb_cls_train_export": (c_int, [c_void_p, POINTER(Weights), c_void_p, c_void_p]),
    "pllb_cls_train_export_grads": (c_int, [c_void_p, POINTER(Weights), c_void_p, c_void_p]),
    "pllb_s2s_create": (c_int, [POINTER(c_void_p), POINTER(S2sDesc), POINTER(S2sWeights), c_int32, c_int]),
    "pllb_s2s_destroy": (c_int, [c_void_p]),
    "pllb_s2s_workspace_bytes": (c_int64, [c_void_p]),
    "pllb_s2s_set_timing": (c_int, [c_void_p, c_int]),
    "pllb_s2s_get_stats": (c_int, [c_void_p, POINTER(S2sStats)]),
    "pllb_s2s_reset_stats": (c_int, [c_void_p]),
    "pllb_generate": (c_int, [c_void_p, POINTER(GenDesc), c_void_p, c_void_p, c_int32, c_void_p, c_void_p, c_void_p,
                              c_void_p]),
    "pllb_generate_host": (c_int, [c_void_p, POINTER(GenDesc), c_void_p, c_void_p, c_int32, c_void_p, c_void_p,
                                   c_void_p]),
    "pllb_generate_beam": (c_int, [c_void_p, POINTER(GenDesc), POINTER(BeamDesc), c_void_p, c_void_p, c_int32, c_void_p,
                                   c_void_p, c_void_p, c_void_p]),
    "pllb_generate_beam_host": (c_int, [c_void_p, POINTER(GenDesc), POINTER(BeamDesc), c_void_p, c_void_p, c_int32,
                                        c_void_p, c_void_p, c_void_p]),
    "pllb_s2s_debug_beam_replay": (c_int, [c_void_p, POINTER(GenDesc), POINTER(BeamDesc), c_int32, c_void_p, c_int32,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "pllb_s2s_train_create": (c_int, [POINTER(c_void_p), POINTER(S2sDesc), POINTER(S2sWeights), POINTER(S2sTrainDesc),
                                      c_int]),
    "pllb_s2s_train_step_host": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32,
                                         POINTER(c_float)]),
    "pllb_s2s_train_export": (c_int, [c_void_p, POINTER(S2sWeights)]),
    "pllb_s2s_train_export_grads": (c_int, [c_void_p, POINTER(S2sWeights)]),
}

_lib = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load libpllb200.so and bind every declared symbol (raises if one is missing)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise FileNotFoundError(f"{LIB_PATH} not built; run `python -c 'import __graft_entry__ as g; g.build()'`")
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.pllb_abi_version() != 1:
        raise RuntimeError("libpllb200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise PllbError(rc, load().pllb_last_error().decode("utf-8", "replace"))


def require_device() -> None:
    if load().pllb_device_count() < 1:
        raise PllbError(3, "no sm_100 (B200) device visible; this package has no CPU fallback")
