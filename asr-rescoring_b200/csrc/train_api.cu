// train_api.cu — C ABI of the MLM fine-tuning path (include/pllb.h, pllb_train_*): replaces the
// train_mode=True branch of run_one_epoch (MLM_PLL/main.py:73-99) — BertForMaskedLM.forward with
// labels, loss.backward(), torch.optim.AdamW.step() — and its loss-only twin (train_mode=False,
// do_scoring=False, the dev pass of mlm_finetune_bert, :146-153).
//
// Numerics: fp32 master parameters, gradients and Adam moments in four flat buffers with one
// layout; every matrix product (forward, dgrad, wgrad) on the tcgen05 GEMM with bf16 operands and
// fp32 accumulation; LayerNorm / softmax / cross entropy / GELU in fp32.  The GEMM takes two
// K-contiguous operands, so a linear layer Y = X W^T keeps W and W^T as bf16 copies (refreshed after
// every optimizer step) and the backward pass transposes dY and X on the fly:
//     dX [R, K] = dY [R, N] . (W^T [K, N])^T          dW [N, K] = dY^T [N, R] . (X^T [K, R])^T
// with R padded to a multiple of 64 by zero columns.  Weight gradients are written by the GEMM
// epilogue straight into the flat gradient buffer.
//
// The same encoder forward / backward also trains the RescoreBert student (pllb_cls_train_*): Linear(H, 1)
// on the [CLS] row in place of the MLM head, with the MD / MWER loss of include/pllb.h.
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

#include "common.h"
#include "train.h"

using namespace pllb;

namespace {

struct Span { int64_t off = 0, n = 0; };

struct TLayer {
  Span qkv_w, qkv_b, ao_w, ao_b, ao_g, ao_be, ff1_w, ff1_b, ff2_w, ff2_b, out_g, out_be;
  __nv_bfloat16 *qkv16, *qkvT16, *ao16, *aoT16, *ff116, *ff1T16, *ff216, *ff2T16;     // operand copies
  // activations kept for the backward pass
  __nv_bfloat16 *x16, *qkv, *ctx, *h1_16, *g16;
  float *lse, *xhat1, *rstd1, *f, *xhat2, *rstd2;
};

enum Site : uint32_t { SITE_EMB = 1, SITE_ATT = 2, SITE_AO = 3, SITE_FF2 = 4 };   // + 8 * layer

// One BART decoder layer of the s2s trainer: causal self-attention + LN, cross-attention + LN, FFN + LN.  The
// cross-attention K / V projections of every layer live in one stacked span of the trainer (ckv_w, ckv_b).
struct DLayer {
  Span qkv_w, qkv_b, o_w, o_b, ln1_g, ln1_b, cq_w, cq_b, co_w, co_b, ln2_g, ln2_b, ff1_w, ff1_b, ff2_w, ff2_b, ln3_g, ln3_b;
  __nv_bfloat16 *qkv16, *qkvT16, *o16, *oT16, *cq16, *cqT16, *co16, *coT16, *ff116, *ff1T16, *ff216, *ff2T16;
  // activations kept for the backward pass
  __nv_bfloat16 *x16, *qkv, *ctx, *h1_16, *cq, *cctx, *h2_16, *g16;
  float *lse, *clse, *xhat1, *rstd1, *xhat2, *rstd2, *f, *xhat3, *rstd3;
};
// dropout sites of the s2s decoder, after the encoder's (8 * layer + 1 .. 4): the embedding at 8 * enc_layers + 1,
// decoder layer l at 8 * (enc_layers + 1 + l) + {SITE_ATT, SITE_AO, SITE_FF2, DSITE_XATT, DSITE_XAO}
enum DSite : uint32_t { DSITE_XATT = 5, DSITE_XAO = 6 };

}  // namespace

struct pllb_trainer_ctx {
  pllb_model_desc d{};
  pllb_train_desc t{};
  int device = 0;
  int Vp = 0;
  int64_t cap_rows = 0, cap_rows_pad = 0;
  std::vector<void*> owned;
  int64_t owned_bytes = 0;
  // flat fp32 buffers, one layout: parameters, gradients, Adam first / second moments
  float *P = nullptr, *G = nullptr, *M = nullptr, *V = nullptr;
  int64_t n_flat = 0;
  Span word, pos, type, emb_g, emb_b, head_w, head_b, head_g, head_be, dec_b;
  std::vector<TLayer> L;
  __nv_bfloat16 *head16 = nullptr, *headT16 = nullptr, *E16 = nullptr, *ET16 = nullptr;
  // batch inputs
  int32_t *ids = nullptr, *labels = nullptr, *n_valid = nullptr;
  int32_t* host_stage = nullptr;     // pinned
  // stash outside the layers
  float *xhat_e = nullptr, *rstd_e = nullptr, *t_f32 = nullptr, *xhat_h = nullptr, *rstd_h = nullptr;
  __nv_bfloat16 *xlast16 = nullptr, *tn16 = nullptr, *dlogits16 = nullptr;
  float *logits = nullptr, *loss_rows = nullptr, *loss_dev = nullptr;
  // scratch
  float *h32 = nullptr, *y32 = nullptr, *dh32 = nullptr, *dz32 = nullptr, *dzd32 = nullptr, *Dq = nullptr, *zeros = nullptr,
        *colsum_scratch = nullptr;
  __nv_bfloat16 *d16 = nullptr, *dT16 = nullptr, *xT16 = nullptr;
  int64_t step = 0;        // optimizer steps since the last reset (Adam bias correction)
  int64_t calls = 0;       // forward passes since create (dropout stream)
  int64_t launches = 0;
  int last_rows = 0;       // B * T of the last step (pllb_train_row_losses_host)
  // per-step scalars (device copy read by the kernels; pinned host copy filled before every step)
  TrainStepParams* params_dev = nullptr;
  TrainStepParams* params_host = nullptr;
  // CUDA graphs of the step, one per (B, T, mode): the step is ~575 small launches (launch-bound at the
  // reference's batch size), all with shape-static arguments.  A shape runs eagerly the first time
  // (shared-memory opt-ins, tensor-map cache), is captured the second time and replayed from then on.
  cudaStream_t stream = nullptr;     // every step runs here (stream capture is not possible on the legacy stream)
  bool use_graph = true;   // PLLB_TRAIN_GRAPH=0 disables
  struct GraphEntry { int seen = 0; cudaGraphExec_t exec = nullptr; int64_t launches = 0; };
  std::unordered_map<uint64_t, GraphEntry> graphs;
  int64_t graph_replays = 0;
  // RescoreBert trainer (pllb_cls_train_create): Linear(H, 1) on the [CLS] row instead of the MLM head.  The flat
  // buffers hold the embeddings, the layers and lin_w / lin_b; there are no head / decoder copies and no logits.
  bool cls = false;
  Span lin_w, lin_b;
  pllb_cls_loss_desc loss{};
  int32_t* group = nullptr;                                                 // [max_rows]
  float *target = nullptr, *am = nullptr, *err = nullptr, *scores = nullptr, *dscore = nullptr;   // [max_rows] each
  // CorrectBart trainer (pllb_s2s_train_create): word = model.shared (Vp rows, rows >= vocab zero), pos / emb_g / emb_b
  // = the encoder's embed_positions (whole table) and layernorm_embedding, L = the encoder layers (BERT form).
  bool s2s = false;
  pllb_s2s_desc sd{};
  int32_t decoder_start_id = 0;
  int cap_batch = 0, cap_enc = 0, cap_dec = 0;
  Span dec_pos, dec_emb_g, dec_emb_b, ckv_w, ckv_b;
  std::vector<DLayer> D;
  __nv_bfloat16 *ckv16 = nullptr, *ckvT16 = nullptr;       // [2H * dec_layers, H] stacked cross K / V weights
  float* flb = nullptr;                                     // final_logits_bias [Vp], a buffer (never updated)
  int32_t* dec_ids = nullptr;                               // shift_tokens_right(labels) [B * T_dec]
  __nv_bfloat16 *ckv = nullptr, *dlast16 = nullptr;         // cross K|V of every layer [B*T_enc, 2H * dec_layers]; decoder output
  float *dckv32 = nullptr, *dq32 = nullptr, *xhat_d = nullptr, *rstd_d = nullptr;
  std::vector<int32_t> dec_host;
};

namespace {

#define RC(expr)            \
  do {                      \
    int _rc = (expr);       \
    if (_rc) return _rc;    \
  } while (0)

template <typename T>
int talloc(pllb_trainer_ctx* c, T** out, int64_t count, bool zero = false) {
  void* p = nullptr;
  const int64_t bytes = std::max<int64_t>(count, 1) * (int64_t)sizeof(T);
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(PLLB_ERR_OOM, "cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
  }
  if (zero) cudaMemset(p, 0, (size_t)bytes);
  c->owned.push_back(p);
  c->owned_bytes += bytes;
  *out = reinterpret_cast<T*>(p);
  return PLLB_OK;
}

Span take(int64_t& cursor, int64_t n) {
  Span s{cursor, n};
  cursor += round_up(n, 64);
  return s;
}

int gemm(const void* A, const void* W, const float* bias, void* C, int64_t M, int N, int K, int epi, cudaStream_t s) {
  return launch_gemm_tcgen05(A, W, bias, C, M, N, K, epi, nullptr, DT_BF16, s);
}

// bf16 copies (row-major and transposed) of one GEMM weight [N, K] of the flat parameter buffer
int refresh_weight(pllb_trainer_ctx* c, Span w, int N, int K, __nv_bfloat16* w16, __nv_bfloat16* wT16, cudaStream_t s) {
  return launch_train_cast_transpose(c->P + w.off, false, N, K, N, w16, wT16, s);
}

int refresh_all(pllb_trainer_ctx* c, cudaStream_t s) {
  const int H = c->d.hidden, I = c->d.intermediate;
  for (auto& l : c->L) {
    RC(refresh_weight(c, l.qkv_w, 3 * H, H, l.qkv16, l.qkvT16, s));
    RC(refresh_weight(c, l.ao_w, H, H, l.ao16, l.aoT16, s));
    RC(refresh_weight(c, l.ff1_w, I, H, l.ff116, l.ff1T16, s));
    RC(refresh_weight(c, l.ff2_w, H, I, l.ff216, l.ff2T16, s));
  }
  if (c->s2s) {
    const int Id = c->sd.dec_intermediate;
    for (auto& l : c->D) {
      RC(refresh_weight(c, l.qkv_w, 3 * H, H, l.qkv16, l.qkvT16, s));
      RC(refresh_weight(c, l.o_w, H, H, l.o16, l.oT16, s));
      RC(refresh_weight(c, l.cq_w, H, H, l.cq16, l.cqT16, s));
      RC(refresh_weight(c, l.co_w, H, H, l.co16, l.coT16, s));
      RC(refresh_weight(c, l.ff1_w, Id, H, l.ff116, l.ff1T16, s));
      RC(refresh_weight(c, l.ff2_w, H, Id, l.ff216, l.ff2T16, s));
    }
    RC(refresh_weight(c, c->ckv_w, 2 * H * c->sd.dec_layers, H, c->ckv16, c->ckvT16, s));
    return refresh_weight(c, c->word, c->Vp, H, c->E16, c->ET16, s);     // the LM head is model.shared
  }
  if (c->cls) return PLLB_OK;     // no MLM head, no tied decoder
  RC(refresh_weight(c, c->head_w, H, H, c->head16, c->headT16, s));
  RC(refresh_weight(c, c->word, c->Vp, H, c->E16, c->ET16, s));
  return PLLB_OK;
}

// dX = dY . W  and  dW = dY^T . X  of one linear layer, plus the bias gradient.
//   dy32 [R, N] fp32 (gradient of the layer's output); x16 [R, K] the layer's bf16 input
//   dx32 [R, K] fp32 out (may be null: the input needs no gradient)
int linear_bwd(pllb_trainer_ctx* c, const float* dy32, const __nv_bfloat16* x16, const __nv_bfloat16* wT16, int R, int N, int K,
               Span w, Span b, float* dx32, cudaStream_t s) {
  const int Rp = (int)round_up(R, 64);
  RC(launch_train_cast_transpose(dy32, false, R, N, Rp, c->d16, c->dT16, s));
  RC(launch_train_colsum(dy32, false, nullptr, R, N, c->G + b.off, nullptr, c->colsum_scratch, s));
  RC(launch_train_cast_transpose(x16, true, R, K, Rp, nullptr, c->xT16, s));
  RC(gemm(c->dT16, c->xT16, c->zeros, c->G + w.off, N, K, Rp, EPI_BIAS_F32, s));            // dW [N, K]
  if (dx32) RC(gemm(c->d16, wT16, c->zeros, dx32, R, K, N, EPI_BIAS_F32, s));                // dX [R, K]
  return PLLB_OK;
}

int copy_in(pllb_trainer_ctx* c, Span dst, const float* src, int64_t n, int64_t dst_off) {
  if (!src)
    return fail(PLLB_ERR_INVALID, c->s2s ? "pllb_s2s_train_create: a weight pointer is null"
                                  : c->cls ? "pllb_cls_train_create: a weight pointer is null"
                                           : "pllb_train_create: a weight pointer is null (the MLM head is required)");
  PLLB_CUDA(cudaMemcpyAsync(c->P + dst.off + dst_off, src, sizeof(float) * n, cudaMemcpyDeviceToDevice, 0));
  return PLLB_OK;
}
int copy_out(const float* buf, Span src, const float* dst, int64_t n, int64_t src_off = 0) {
  if (!dst) return PLLB_OK;
  PLLB_CUDA(cudaMemcpyAsync(const_cast<float*>(dst), buf + src.off + src_off, sizeof(float) * n, cudaMemcpyDeviceToDevice, 0));
  return PLLB_OK;
}

// The encoder layers of w, in the trainer's flat layout (q / k / v stacked in qkv_w and qkv_b).
template <typename Fn>
int visit_enc_layers(const pllb_trainer_ctx* c, const pllb_weights* w, Fn fn) {
  const int H = c->d.hidden, I = c->d.intermediate;
  const int64_t HH = (int64_t)H * H;
  for (int l = 0; l < c->d.num_layers; ++l) {
    const pllb_layer_weights& lw = w->layers[l];
    const TLayer& t = c->L[l];
    RC(fn(t.qkv_w, lw.q_w, HH, 0)); RC(fn(t.qkv_w, lw.k_w, HH, HH)); RC(fn(t.qkv_w, lw.v_w, HH, 2 * HH));
    RC(fn(t.qkv_b, lw.q_b, H, 0)); RC(fn(t.qkv_b, lw.k_b, H, H)); RC(fn(t.qkv_b, lw.v_b, H, 2 * H));
    RC(fn(t.ao_w, lw.ao_w, HH, 0)); RC(fn(t.ao_b, lw.ao_b, H, 0));
    RC(fn(t.ao_g, lw.ao_ln_g, H, 0)); RC(fn(t.ao_be, lw.ao_ln_b, H, 0));
    RC(fn(t.ff1_w, lw.ff1_w, (int64_t)I * H, 0)); RC(fn(t.ff1_b, lw.ff1_b, I, 0));
    RC(fn(t.ff2_w, lw.ff2_w, (int64_t)H * I, 0)); RC(fn(t.ff2_b, lw.ff2_b, H, 0));
    RC(fn(t.out_g, lw.out_ln_g, H, 0)); RC(fn(t.out_be, lw.out_ln_b, H, 0));
  }
  return PLLB_OK;
}

// Every tensor of a BART trainer in one fixed order: shared, the encoder's positions / layernorm_embedding / layers,
// the decoder's positions / layernorm_embedding / layers.  Cross K and V of decoder layer l go to rows
// [2H l, 2H l + H) and [2H l + H, 2H (l + 1)) of ckv_w (and the same entries of ckv_b).  final_logits_bias is not a
// parameter and is not visited.
template <typename Fn>
int visit_s2s_params(const pllb_trainer_ctx* c, const pllb_s2s_weights* w, Fn fn) {
  const pllb_s2s_desc& sd = c->sd;
  const int H = sd.hidden, Id = sd.dec_intermediate;
  const int64_t HH = (int64_t)H * H;
  RC(fn(c->word, w->shared, (int64_t)sd.vocab * H, 0));
  RC(fn(c->pos, w->enc.pos_emb, (int64_t)(sd.enc_max_position + 2) * H, 0));
  RC(fn(c->emb_g, w->enc.emb_ln_g, H, 0));
  RC(fn(c->emb_b, w->enc.emb_ln_b, H, 0));
  RC(visit_enc_layers(c, &w->enc, fn));
  RC(fn(c->dec_pos, w->dec_pos_emb, (int64_t)(sd.dec_max_position + 2) * H, 0));
  RC(fn(c->dec_emb_g, w->dec_emb_ln_g, H, 0));
  RC(fn(c->dec_emb_b, w->dec_emb_ln_b, H, 0));
  for (int l = 0; l < sd.dec_layers; ++l) {
    const pllb_dec_layer_weights& lw = w->dec_layers[l];
    const DLayer& t = c->D[l];
    RC(fn(t.qkv_w, lw.q_w, HH, 0)); RC(fn(t.qkv_w, lw.k_w, HH, HH)); RC(fn(t.qkv_w, lw.v_w, HH, 2 * HH));
    RC(fn(t.qkv_b, lw.q_b, H, 0)); RC(fn(t.qkv_b, lw.k_b, H, H)); RC(fn(t.qkv_b, lw.v_b, H, 2 * H));
    RC(fn(t.o_w, lw.o_w, HH, 0)); RC(fn(t.o_b, lw.o_b, H, 0));
    RC(fn(t.ln1_g, lw.self_ln_g, H, 0)); RC(fn(t.ln1_b, lw.self_ln_b, H, 0));
    RC(fn(t.cq_w, lw.cq_w, HH, 0)); RC(fn(t.cq_b, lw.cq_b, H, 0));
    RC(fn(c->ckv_w, lw.ck_w, HH, 2 * l * HH)); RC(fn(c->ckv_w, lw.cv_w, HH, (2 * l + 1) * HH));
    RC(fn(c->ckv_b, lw.ck_b, H, 2 * l * H)); RC(fn(c->ckv_b, lw.cv_b, H, (2 * l + 1) * H));
    RC(fn(t.co_w, lw.co_w, HH, 0)); RC(fn(t.co_b, lw.co_b, H, 0));
    RC(fn(t.ln2_g, lw.cross_ln_g, H, 0)); RC(fn(t.ln2_b, lw.cross_ln_b, H, 0));
    RC(fn(t.ff1_w, lw.ff1_w, (int64_t)Id * H, 0)); RC(fn(t.ff1_b, lw.ff1_b, Id, 0));
    RC(fn(t.ff2_w, lw.ff2_w, (int64_t)H * Id, 0)); RC(fn(t.ff2_b, lw.ff2_b, H, 0));
    RC(fn(t.ln3_g, lw.final_ln_g, H, 0)); RC(fn(t.ln3_b, lw.final_ln_b, H, 0));
  }
  return PLLB_OK;
}

// Every external tensor of a trainer with its place in the flat buffers, in one fixed order: the embeddings, the
// layers (q / k / v stacked in qkv_w and qkv_b), then the MLM head or lin_w / lin_b.  fn(span, ext, n, off) moves the
// n floats of `ext` to or from span offset `off`.  The word embedding is V x H floats: rows >= vocab of the padded
// MLM span are not part of any tensor.  The tied decoder weight is not visited.
template <typename Fn>
int visit_params(const pllb_trainer_ctx* c, const pllb_weights* w, const float* lin_w, const float* lin_b, Fn fn) {
  const int H = c->d.hidden, V = c->d.vocab;
  const int64_t HH = (int64_t)H * H;
  RC(fn(c->word, w->word_emb, (int64_t)V * H, 0));
  RC(fn(c->pos, w->pos_emb, (int64_t)c->d.max_position * H, 0));
  RC(fn(c->type, w->type_emb, 2 * H, 0));
  RC(fn(c->emb_g, w->emb_ln_g, H, 0));
  RC(fn(c->emb_b, w->emb_ln_b, H, 0));
  RC(visit_enc_layers(c, w, fn));
  if (c->cls) {
    RC(fn(c->lin_w, lin_w, H, 0)); RC(fn(c->lin_b, lin_b, 1, 0));
  } else {
    RC(fn(c->head_w, w->head_w, HH, 0)); RC(fn(c->head_b, w->head_b, H, 0));
    RC(fn(c->head_g, w->head_ln_g, H, 0)); RC(fn(c->head_be, w->head_ln_b, H, 0));
    RC(fn(c->dec_b, w->decoder_b, V, 0));
  }
  return PLLB_OK;
}

// drop probability p (0: no dropout) over the DEVICE seed; shared by the trainers and the kernel test hooks
TrainDrop drop_of(const uint64_t* seed, float p) {
  TrainDrop d{};
  d.seed = seed;
  if (p > 0.f) {
    d.thresh = (uint32_t)std::min<double>(4294967295.0, (double)p * 4294967296.0);
    d.inv_keep = 1.f / (1.f - p);
  } else {
    d.thresh = 0;
    d.inv_keep = 1.f;
  }
  return d;
}

TrainDrop make_drop(const pllb_trainer_ctx* c, float p, bool train) {
  return drop_of(&c->params_dev->seed, train ? p : 0.f);
}

// The encoder forward of one step: embeddings and every layer.  On return h32 holds the fp32 output of the
// last layer (and xlast16 its bf16 copy, when the trainer has an MLM head to feed).
int encoder_fwd(pllb_trainer_ctx* c, int B, int T, const TrainDrop& hd, const TrainDrop& ad, cudaStream_t s) {
  const pllb_model_desc& d = c->d;
  const int H = d.hidden, I = d.intermediate, NH = d.num_heads, NL = d.num_layers;
  const int R = B * T;
  float* P = c->P;
  if (c->s2s)
    RC(launch_train_bart_embed(c->ids, T, P + c->word.off, c->sd.embed_scale, P + c->pos.off + 2 * H, P + c->emb_g.off,
                               P + c->emb_b.off, d.ln_eps, R, H, hd, SITE_EMB, c->h32, c->L[0].x16, c->xhat_e, c->rstd_e, s));
  else
    RC(launch_train_embed(c->ids, T, P + c->word.off, P + c->pos.off, P + c->type.off, P + c->emb_g.off, P + c->emb_b.off,
                          d.ln_eps, R, H, hd, SITE_EMB, c->h32, NL > 0 ? (void*)c->L[0].x16 : (void*)c->xlast16, c->xhat_e,
                          c->rstd_e, s));
  for (int l = 0; l < NL; ++l) {
    TLayer& t = c->L[l];
    __nv_bfloat16* x_next = l + 1 < NL ? c->L[l + 1].x16 : c->xlast16;
    RC(gemm(t.x16, t.qkv16, P + t.qkv_b.off, t.qkv, R, 3 * H, H, EPI_BIAS_BF16, s));
    RC(launch_train_attn_fwd(t.qkv, c->n_valid, R, T, H, NH, ad, SITE_ATT + 8 * l, t.ctx, t.lse, s));
    RC(gemm(t.ctx, t.ao16, P + t.ao_b.off, c->y32, R, H, H, EPI_BIAS_F32, s));
    RC(launch_train_ln_fwd(c->y32, c->h32, P + t.ao_g.off, P + t.ao_be.off, d.ln_eps, R, H, hd, SITE_AO + 8 * l, c->h32,
                           t.h1_16, t.xhat1, t.rstd1, s));
    RC(gemm(t.h1_16, t.ff116, P + t.ff1_b.off, t.f, R, I, H, EPI_BIAS_F32, s));
    RC(launch_train_gelu_fwd(t.f, (int64_t)R * I, t.g16, nullptr, s));
    RC(gemm(t.g16, t.ff216, P + t.ff2_b.off, c->y32, R, H, I, EPI_BIAS_F32, s));
    RC(launch_train_ln_fwd(c->y32, c->h32, P + t.out_g.off, P + t.out_be.off, d.ln_eps, R, H, hd, SITE_FF2 + 8 * l, c->h32,
                           x_next, t.xhat2, t.rstd2, s));
  }
  return PLLB_OK;
}

// The encoder backward of one step, from dh32 = gradient of the last layer's output (written by the head's
// backward) down to the embedding gradients.  The word-embedding gradient is ADDED to G[word] (the MLM head
// has written the tied decoder's part there; a CLS trainer clears it first).
int encoder_bwd(pllb_trainer_ctx* c, int B, int T, const TrainDrop& hd, const TrainDrop& ad, cudaStream_t s) {
  const pllb_model_desc& d = c->d;
  const int H = d.hidden, I = d.intermediate, NH = d.num_heads, NL = d.num_layers;
  const int R = B * T;
  float* P = c->P;
  float* G = c->G;
  // dh32 = gradient of the layer output through the layer above; dz32 = the part that arrives over the
  // residual connection (added inside ln_bwd)
  bool have_res = false;
  for (int l = NL - 1; l >= 0; --l) {
    TLayer& t = c->L[l];
    const bool dr = hd.thresh != 0;
    // BertOutput: LN(dropout(FFN2(g)) + h1)
    RC(launch_train_ln_bwd(c->dh32, have_res ? c->dz32 : nullptr, P + t.out_g.off, t.xhat2, t.rstd2, R, H, hd, -1,
                           dr ? (int)(SITE_FF2 + 8 * l) : -1, c->dz32, dr ? c->dzd32 : nullptr, s));
    RC(launch_train_colsum(c->dh32, false, t.xhat2, R, H, G + t.out_be.off, G + t.out_g.off, c->colsum_scratch, s));
    RC(linear_bwd(c, dr ? c->dzd32 : c->dz32, t.g16, t.ff2T16, R, H, I, t.ff2_w, t.ff2_b, c->y32, s));   // y32 = dg [R, I]
    RC(launch_train_gelu_bwd(c->y32, t.f, (int64_t)R * I, s));
    RC(linear_bwd(c, c->y32, t.h1_16, t.ff1T16, R, I, H, t.ff1_w, t.ff1_b, c->dh32, s));                 // dh32 = dh1 via the FFN
    // BertSelfOutput: LN(dropout(AO(ctx)) + x)
    RC(launch_train_ln_bwd(c->dh32, c->dz32, P + t.ao_g.off, t.xhat1, t.rstd1, R, H, hd, -1,
                           dr ? (int)(SITE_AO + 8 * l) : -1, c->dz32, dr ? c->dzd32 : nullptr, s));
    RC(launch_train_colsum(c->dh32, false, t.xhat1, R, H, G + t.ao_be.off, G + t.ao_g.off, c->colsum_scratch, s));
    RC(linear_bwd(c, dr ? c->dzd32 : c->dz32, t.ctx, t.aoT16, R, H, H, t.ao_w, t.ao_b, c->dh32, s));     // dh32 = dctx
    RC(launch_train_attn_bwd(t.qkv, c->dh32, t.lse, c->n_valid, R, T, H, NH, ad, SITE_ATT + 8 * l, c->y32, c->Dq, s));
    RC(linear_bwd(c, c->y32, t.x16, t.qkvT16, R, 3 * H, H, t.qkv_w, t.qkv_b, c->dh32, s));               // dh32 = dx via QKV
    have_res = true;
  }
  // embeddings (dropout sits AFTER the LayerNorm here)
  RC(launch_train_ln_bwd(c->dh32, have_res ? c->dz32 : nullptr, P + c->emb_g.off, c->xhat_e, c->rstd_e, R, H, hd,
                         hd.thresh != 0 ? (int)SITE_EMB : -1, -1, c->dz32, nullptr, s));
  RC(launch_train_colsum(c->dh32, false, c->xhat_e, R, H, G + c->emb_b.off, G + c->emb_g.off, c->colsum_scratch, s));
  if (c->s2s)      // adds to G[shared] after the LM head and the decoder lookup
    return launch_train_bart_embed_bwd(c->dz32, c->ids, B, T, H, d.max_position, c->t.pad_id, c->sd.embed_scale,
                                       G + c->word.off, G + c->pos.off + 2 * H, s);
  RC(launch_train_embed_bwd(c->dz32, c->ids, B, T, H, d.max_position, c->t.pad_id, G + c->word.off, G + c->pos.off,
                            G + c->type.off, c->colsum_scratch, s));
  return PLLB_OK;
}

int optimizer_update(pllb_trainer_ctx* c, cudaStream_t s) {
  RC(launch_train_adamw(c->P, c->G, c->M, c->V, c->n_flat, c->t.lr, c->t.beta1, c->t.beta2, c->t.adam_eps,
                        c->t.weight_decay, c->params_dev, s));
  return refresh_all(c, s);
}

// Every launch of one MLM step (shape-static arguments only; the per-step scalars are read from params_dev).
// mode 0: loss only (model.eval()); 1: forward + backward + AdamW step; 2: forward + backward, no update
int enqueue_mlm_step(pllb_trainer_ctx* c, int B, int T, int mode, cudaStream_t s) {
  const pllb_model_desc& d = c->d;
  const int H = d.hidden, Vp = c->Vp, V = d.vocab;
  const int R = B * T, Rp = (int)round_up(R, 64);
  const bool train = mode != 0;
  const TrainDrop hd = make_drop(c, c->t.hidden_dropout, train), ad = make_drop(c, c->t.attention_dropout, train);
  float* P = c->P;
  RC(encoder_fwd(c, B, T, hd, ad, s));
  // MLM head on EVERY row (labels are the whole sequence, MLM_PLL/preprocess.py:24-28)
  RC(gemm(c->xlast16, c->head16, P + c->head_b.off, c->t_f32, R, H, H, EPI_BIAS_F32, s));
  RC(launch_train_gelu_fwd(c->t_f32, (int64_t)R * H, nullptr, c->y32, s));
  TrainDrop none{&c->params_dev->seed, 0, 1.f};
  RC(launch_train_ln_fwd(c->y32, nullptr, P + c->head_g.off, P + c->head_be.off, d.ln_eps, R, H, none, 0, nullptr, c->tn16,
                         c->xhat_h, c->rstd_h, s));
  RC(gemm(c->tn16, c->E16, P + c->dec_b.off, c->logits, R, Vp, H, EPI_BIAS_F32, s));
  RC(launch_train_ce(c->logits, c->labels, R, V, Vp, c->loss_rows, train ? c->dlogits16 : nullptr, c->loss_dev, s));
  if (train) {
    float* G = c->G;
    // ---------------- backward: head
    RC(launch_train_cast_transpose(c->dlogits16, true, R, Vp, Rp, nullptr, c->dT16, s));
    const float inv_r = 1.f / (float)R;        // the mean over the B*T positions, applied in fp32 (ce_kernel)
    RC(launch_train_colsum(c->dlogits16, true, nullptr, R, Vp, G + c->dec_b.off, nullptr, c->colsum_scratch, s));
    RC(launch_train_scale(G + c->dec_b.off, Vp, inv_r, s));
    RC(launch_train_cast_transpose(c->tn16, true, R, H, Rp, nullptr, c->xT16, s));
    RC(gemm(c->dT16, c->xT16, c->zeros, G + c->word.off, Vp, H, Rp, EPI_BIAS_F32, s));       // decoder part of dE
    RC(launch_train_scale(G + c->word.off, (int64_t)Vp * H, inv_r, s));
    RC(gemm(c->dlogits16, c->ET16, c->zeros, c->dh32, R, H, Vp, EPI_BIAS_F32, s));           // d(transform LayerNorm output)
    RC(launch_train_scale(c->dh32, (int64_t)R * H, inv_r, s));
    RC(launch_train_ln_bwd(c->dh32, nullptr, P + c->head_g.off, c->xhat_h, c->rstd_h, R, H, none, -1, -1, c->dz32, nullptr, s));
    RC(launch_train_colsum(c->dh32, false, c->xhat_h, R, H, G + c->head_be.off, G + c->head_g.off, c->colsum_scratch, s));
    RC(launch_train_gelu_bwd(c->dz32, c->t_f32, (int64_t)R * H, s));
    RC(linear_bwd(c, c->dz32, c->xlast16, c->headT16, R, H, H, c->head_w, c->head_b, c->dh32, s));
    // ---------------- backward: encoder
    RC(encoder_bwd(c, B, T, hd, ad, s));
    if (mode == 1) RC(optimizer_update(c, s));
  }
  return PLLB_OK;
}

// Every launch of one RescoreBert step: the same encoder, the Linear(H, 1) head on the [CLS] rows, the MD / MWER
// loss over the per-hypothesis scores.  The batch's targets, AM scores, errors and group indices are read from
// device memory, so the graph of a (B, T, mode) serves every batch of that shape.
int enqueue_cls_step(pllb_trainer_ctx* c, int B, int T, int mode, cudaStream_t s) {
  const int H = c->d.hidden;
  const bool train = mode != 0;
  const TrainDrop hd = make_drop(c, c->t.hidden_dropout, train), ad = make_drop(c, c->t.attention_dropout, train);
  float* P = c->P;
  float* G = c->G;
  RC(encoder_fwd(c, B, T, hd, ad, s));
  RC(launch_train_cls_fwd(c->h32, P + c->lin_w.off, P + c->lin_b.off, B, T, H, c->scores, s));
  RC(launch_train_cls_loss(c->scores, c->target, c->am, c->err, c->group, B, c->loss.md_weight, c->loss.mwer_weight,
                           c->loss.am_weight, train ? c->dscore : nullptr, c->loss_dev, s));
  if (train) {
    RC(launch_train_cls_bwd(c->h32, P + c->lin_w.off, c->dscore, B, T, H, G + c->lin_w.off, G + c->lin_b.off, c->dh32, s));
    // no tied decoder: the embedding scatter adds to a cleared word-embedding gradient
    PLLB_CUDA(cudaMemsetAsync(G + c->word.off, 0, sizeof(float) * (size_t)c->word.n, s));
    RC(encoder_bwd(c, B, T, hd, ad, s));
    if (mode == 1) RC(optimizer_update(c, s));
  }
  return PLLB_OK;
}

uint32_t dsite(const pllb_trainer_ctx* c, int l, uint32_t k) { return 8u * (uint32_t)(c->sd.enc_layers + 1 + l) + k; }

// Every launch of one CorrectBart step (BartForConditionalGeneration.forward with labels): the encoder, the cross K|V
// of every decoder layer in one GEMM, the decoder layers, the LM head over shared (Vp columns) + final_logits_bias,
// cross entropy with ignore_index; then the backward in reverse and AdamW.  The 1 / N of the mean (N = labelled
// positions) is read from device memory (loss_dev[1]), so the graph of a (B, T_enc, T_dec, mode) serves every batch
// of that shape.
int enqueue_s2s_step(pllb_trainer_ctx* c, int B, int Te, int Td, int mode, cudaStream_t s) {
  const pllb_s2s_desc& sd = c->sd;
  const int H = sd.hidden, NH = sd.num_heads, NL = sd.dec_layers, Id = sd.dec_intermediate, Vp = c->Vp, V = sd.vocab;
  const int Re = B * Te, Rd = B * Td, Rdp = (int)round_up(Rd, 64), KV = 2 * H * NL;
  const float eps = sd.ln_eps, scale = sd.embed_scale;
  const bool train = mode != 0;
  const TrainDrop hd = make_drop(c, c->t.hidden_dropout, train), ad = make_drop(c, c->t.attention_dropout, train);
  const uint32_t emb_site = 8u * (uint32_t)sd.enc_layers + SITE_EMB;
  float* P = c->P;
  RC(encoder_fwd(c, B, Te, hd, ad, s));                                                    // xlast16 = encoder output
  RC(gemm(c->xlast16, c->ckv16, P + c->ckv_b.off, c->ckv, Re, KV, H, EPI_BIAS_BF16, s));
  RC(launch_train_bart_embed(c->dec_ids, Td, P + c->word.off, scale, P + c->dec_pos.off + 2 * H, P + c->dec_emb_g.off,
                             P + c->dec_emb_b.off, eps, Rd, H, hd, emb_site, c->h32, c->D[0].x16, c->xhat_d, c->rstd_d, s));
  std::vector<S2sAttn> self(NL), cross(NL);
  for (int l = 0; l < NL; ++l) {
    DLayer& t = c->D[l];
    __nv_bfloat16* x_next = l + 1 < NL ? c->D[l + 1].x16 : c->dlast16;
    self[l] = S2sAttn{t.qkv, t.qkv + H, t.qkv + 2 * H, 3 * H, 3 * H, B, Td, Td, NH, true, nullptr};
    cross[l] = S2sAttn{t.cq, c->ckv + (size_t)2 * H * l, c->ckv + (size_t)2 * H * l + H, H, KV, B, Td, Te, NH, false, c->n_valid};
    RC(gemm(t.x16, t.qkv16, P + t.qkv_b.off, t.qkv, Rd, 3 * H, H, EPI_BIAS_BF16, s));
    RC(launch_train_attn_s2s_fwd(self[l], ad, dsite(c, l, SITE_ATT), t.ctx, t.lse, s));
    RC(gemm(t.ctx, t.o16, P + t.o_b.off, c->y32, Rd, H, H, EPI_BIAS_F32, s));
    RC(launch_train_ln_fwd(c->y32, c->h32, P + t.ln1_g.off, P + t.ln1_b.off, eps, Rd, H, hd, dsite(c, l, SITE_AO), c->h32,
                           t.h1_16, t.xhat1, t.rstd1, s));
    RC(gemm(t.h1_16, t.cq16, P + t.cq_b.off, t.cq, Rd, H, H, EPI_BIAS_BF16, s));
    RC(launch_train_attn_s2s_fwd(cross[l], ad, dsite(c, l, DSITE_XATT), t.cctx, t.clse, s));
    RC(gemm(t.cctx, t.co16, P + t.co_b.off, c->y32, Rd, H, H, EPI_BIAS_F32, s));
    RC(launch_train_ln_fwd(c->y32, c->h32, P + t.ln2_g.off, P + t.ln2_b.off, eps, Rd, H, hd, dsite(c, l, DSITE_XAO), c->h32,
                           t.h2_16, t.xhat2, t.rstd2, s));
    RC(gemm(t.h2_16, t.ff116, P + t.ff1_b.off, t.f, Rd, Id, H, EPI_BIAS_F32, s));
    RC(launch_train_gelu_fwd(t.f, (int64_t)Rd * Id, t.g16, nullptr, s));
    RC(gemm(t.g16, t.ff216, P + t.ff2_b.off, c->y32, Rd, H, Id, EPI_BIAS_F32, s));
    RC(launch_train_ln_fwd(c->y32, c->h32, P + t.ln3_g.off, P + t.ln3_b.off, eps, Rd, H, hd, dsite(c, l, SITE_FF2), c->h32,
                           x_next, t.xhat3, t.rstd3, s));
  }
  RC(gemm(c->dlast16, c->E16, c->flb, c->logits, Rd, Vp, H, EPI_BIAS_F32, s));
  RC(launch_train_ce_ignore(c->logits, c->labels, Rd, V, Vp, c->loss_rows, train ? c->dlogits16 : nullptr, c->loss_dev, s));
  if (!train) return PLLB_OK;
  float* G = c->G;
  const float* inv_n = c->loss_dev + 1;
  // ---------------- backward: LM head (writes G[shared] first; final_logits_bias gets nothing)
  RC(launch_train_cast_transpose(c->dlogits16, true, Rd, Vp, Rdp, nullptr, c->dT16, s));
  RC(launch_train_cast_transpose(c->dlast16, true, Rd, H, Rdp, nullptr, c->xT16, s));
  RC(gemm(c->dT16, c->xT16, c->zeros, G + c->word.off, Vp, H, Rdp, EPI_BIAS_F32, s));
  RC(launch_train_scale_dev(G + c->word.off, (int64_t)Vp * H, inv_n, s));
  RC(gemm(c->dlogits16, c->ET16, c->zeros, c->dh32, Rd, H, Vp, EPI_BIAS_F32, s));
  RC(launch_train_scale_dev(c->dh32, (int64_t)Rd * H, inv_n, s));
  // ---------------- backward: decoder layers (dz32 = the part arriving over the residual connection)
  const bool dr = hd.thresh != 0;
  float* dres = dr ? c->dzd32 : c->dz32;      // gradient of the GEMM output that went through dropout
  for (int l = NL - 1; l >= 0; --l) {
    DLayer& t = c->D[l];
    // FFN: LN(dropout(fc2(gelu(fc1(h2)))) + h2)
    RC(launch_train_ln_bwd(c->dh32, l + 1 < NL ? c->dz32 : nullptr, P + t.ln3_g.off, t.xhat3, t.rstd3, Rd, H, hd, -1,
                           dr ? (int)dsite(c, l, SITE_FF2) : -1, c->dz32, dr ? c->dzd32 : nullptr, s));
    RC(launch_train_colsum(c->dh32, false, t.xhat3, Rd, H, G + t.ln3_b.off, G + t.ln3_g.off, c->colsum_scratch, s));
    RC(linear_bwd(c, dres, t.g16, t.ff2T16, Rd, H, Id, t.ff2_w, t.ff2_b, c->y32, s));
    RC(launch_train_gelu_bwd(c->y32, t.f, (int64_t)Rd * Id, s));
    RC(linear_bwd(c, c->y32, t.h2_16, t.ff1T16, Rd, Id, H, t.ff1_w, t.ff1_b, c->dh32, s));
    // cross-attention: LN(dropout(out(attn(q(h1), K|V(enc)))) + h1); dK|dV of this layer into its columns of dckv32
    RC(launch_train_ln_bwd(c->dh32, c->dz32, P + t.ln2_g.off, t.xhat2, t.rstd2, Rd, H, hd, -1,
                           dr ? (int)dsite(c, l, DSITE_XAO) : -1, c->dz32, dr ? c->dzd32 : nullptr, s));
    RC(launch_train_colsum(c->dh32, false, t.xhat2, Rd, H, G + t.ln2_b.off, G + t.ln2_g.off, c->colsum_scratch, s));
    RC(linear_bwd(c, dres, t.cctx, t.coT16, Rd, H, H, t.co_w, t.co_b, c->dh32, s));                    // dh32 = dcctx
    RC(launch_train_attn_s2s_bwd(cross[l], c->dh32, t.clse, ad, dsite(c, l, DSITE_XATT), c->dq32, H,
                                 c->dckv32 + (size_t)2 * H * l, c->dckv32 + (size_t)2 * H * l + H, KV, c->Dq, s));
    RC(linear_bwd(c, c->dq32, t.h1_16, t.cqT16, Rd, H, H, t.cq_w, t.cq_b, c->dh32, s));                // dh32 = dh1 via q
    // causal self-attention: LN(dropout(out(attn(qkv(x)))) + x)
    RC(launch_train_ln_bwd(c->dh32, c->dz32, P + t.ln1_g.off, t.xhat1, t.rstd1, Rd, H, hd, -1,
                           dr ? (int)dsite(c, l, SITE_AO) : -1, c->dz32, dr ? c->dzd32 : nullptr, s));
    RC(launch_train_colsum(c->dh32, false, t.xhat1, Rd, H, G + t.ln1_b.off, G + t.ln1_g.off, c->colsum_scratch, s));
    RC(linear_bwd(c, dres, t.ctx, t.oT16, Rd, H, H, t.o_w, t.o_b, c->dh32, s));                         // dh32 = dctx
    RC(launch_train_attn_s2s_bwd(self[l], c->dh32, t.lse, ad, dsite(c, l, SITE_ATT), c->y32, 3 * H, c->y32 + H,
                                 c->y32 + 2 * H, 3 * H, c->Dq, s));
    RC(linear_bwd(c, c->y32, t.x16, t.qkvT16, Rd, 3 * H, H, t.qkv_w, t.qkv_b, c->dh32, s));           // dh32 = dx
  }
  // decoder embeddings (dropout after the LayerNorm); the lookup adds to G[shared]
  RC(launch_train_ln_bwd(c->dh32, c->dz32, P + c->dec_emb_g.off, c->xhat_d, c->rstd_d, Rd, H, hd, dr ? (int)emb_site : -1, -1,
                         c->dz32, nullptr, s));
  RC(launch_train_colsum(c->dh32, false, c->xhat_d, Rd, H, G + c->dec_emb_b.off, G + c->dec_emb_g.off, c->colsum_scratch, s));
  RC(launch_train_bart_embed_bwd(c->dz32, c->dec_ids, B, Td, H, sd.dec_max_position, c->t.pad_id, scale, G + c->word.off,
                                 G + c->dec_pos.off + 2 * H, s));
  // cross K|V of every layer: one dgrad GEMM sums the layers' contributions to d(encoder output) in layer order
  RC(linear_bwd(c, c->dckv32, c->xlast16, c->ckvT16, Re, KV, H, c->ckv_w, c->ckv_b, c->dh32, s));
  RC(encoder_bwd(c, B, Te, hd, ad, s));
  if (mode == 1) RC(optimizer_update(c, s));
  return PLLB_OK;
}

int enqueue(pllb_trainer_ctx* c, int B, int T, int T2, int mode, cudaStream_t s) {
  if (c->s2s) return enqueue_s2s_step(c, B, T, T2, mode, s);
  return c->cls ? enqueue_cls_step(c, B, T, mode, s) : enqueue_mlm_step(c, B, T, mode, s);
}

// T2: the decoder length of an s2s step (0 otherwise); one graph per (B, T, T2, mode)
int step_impl(pllb_trainer_ctx* c, int B, int T, int mode, float* out_loss_host, cudaStream_t s, int T2 = 0) {
  // per-step scalars -> device (the previous step ended with a stream synchronise, so the pinned copy is free)
  c->calls += 1;
  if (mode == 1) c->step += 1;
  const int64_t t = std::max<int64_t>(c->step, 1);
  const double bc1 = 1.0 - std::pow((double)c->t.beta1, (double)t), bc2 = 1.0 - std::pow((double)c->t.beta2, (double)t);
  c->params_host->seed = c->t.seed * 0x9E3779B97F4A7C15ull + (uint64_t)c->calls * 0xC2B2AE3D27D4EB4Full;
  c->params_host->adam_step_size = (float)((double)c->t.lr / bc1);
  c->params_host->adam_bc2_sqrt = (float)std::sqrt(bc2);
  PLLB_CUDA(cudaMemcpyAsync(c->params_dev, c->params_host, sizeof(TrainStepParams), cudaMemcpyHostToDevice, s));
  const uint64_t key = c->s2s ? ((uint64_t)(uint32_t)B << 42) | ((uint64_t)(uint32_t)T << 22) | ((uint64_t)(uint32_t)T2 << 2) | (uint64_t)mode
                              : ((uint64_t)(uint32_t)B << 34) | ((uint64_t)(uint32_t)T << 2) | (uint64_t)mode;
  pllb_trainer_ctx::GraphEntry* ge = c->use_graph ? &c->graphs[key] : nullptr;
  if (ge && ge->exec) {
    PLLB_CUDA(cudaGraphLaunch(ge->exec, s));
    c->launches += ge->launches;
    c->graph_replays += 1;
  } else if (ge && ge->seen >= 1) {
    if (c->graphs.size() > 256) {              // bound the cache (a caller that never repeats a shape): start over
      for (auto& kv : c->graphs)
        if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
      c->graphs.clear();
      ge = &c->graphs[key];
      ge->seen = 1;
    }
    const int64_t before = g_launch_counter;
    PLLB_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue(c, B, T, T2, mode, s);
    cudaGraph_t g = nullptr;
    const cudaError_t e = cudaStreamEndCapture(s, &g);
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (e != cudaSuccess || !g) return fail(PLLB_ERR_CUDA, std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ei = cudaGraphInstantiate(&exec, g, 0);
    cudaGraphDestroy(g);
    if (ei != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ei));
    ge->exec = exec;
    ge->launches = g_launch_counter - before;
    PLLB_CUDA(cudaGraphLaunch(ge->exec, s));
    c->launches += ge->launches;
    c->graph_replays += 1;
  } else {
    const int64_t before = g_launch_counter;
    RC(enqueue(c, B, T, T2, mode, s));
    c->launches += g_launch_counter - before;
    if (ge) ge->seen += 1;
  }
  if (out_loss_host) {
    PLLB_CUDA(cudaMemcpyAsync(out_loss_host, c->loss_dev, sizeof(float), cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaStreamSynchronize(s));
  }
  return PLLB_OK;
}

enum Kind { KIND_MLM, KIND_CLS, KIND_S2S };
Kind kind_of(const pllb_trainer_ctx* c) { return c->s2s ? KIND_S2S : c->cls ? KIND_CLS : KIND_MLM; }

// `who` takes trainers of kind k (k2 too when given); any other kind is PLLB_ERR_INVALID
int require_kind(const pllb_trainer_ctx* c, Kind k, const char* who, int k2 = -1) {
  if (!c) return fail(PLLB_ERR_INVALID, std::string(who) + ": null trainer");
  const Kind ck = kind_of(c);
  if (ck == k || (int)ck == k2) return PLLB_OK;
  static const char* takes[] = {": an MLM trainer takes pllb_train_step_host / _row_losses_host / _export / _export_grads",
                                ": a RescoreBert trainer takes pllb_cls_train_step_host / _export / _export_grads",
                                ": a CorrectBart trainer takes pllb_s2s_train_step_host / _export / _export_grads and "
                                "pllb_train_row_losses_host"};
  return fail(PLLB_ERR_INVALID, std::string(who) + takes[ck]);
}

// state_dict tensors (and lin_w / lin_b of a RescoreBert trainer) <- the parameters or the gradients
int export_params(pllb_trainer c, bool cls, bool grads, const pllb_weights* w, const float* lin_w, const float* lin_b,
                  const char* who) {
  if (!c || !w || !w->layers) return fail(PLLB_ERR_INVALID, std::string(who) + ": null argument");
  RC(require_kind(c, cls ? KIND_CLS : KIND_MLM, who));
  const float* buf = grads ? c->G : c->P;
  PLLB_CUDA(cudaSetDevice(c->device));
  PLLB_CUDA(cudaStreamSynchronize(c->stream));
  RC(visit_params(c, w, lin_w, lin_b,
                  [buf](Span s, const float* dst, int64_t n, int64_t off) { return copy_out(buf, s, dst, n, off); }));
  // the decoder weight is the word-embedding matrix (tied): written only when the caller keeps a separate tensor
  if (!c->cls && w->decoder_w && w->decoder_w != w->word_emb)
    RC(copy_out(buf, c->word, w->decoder_w, (int64_t)c->d.vocab * c->d.hidden));
  PLLB_CUDA(cudaStreamSynchronize(0));
  return PLLB_OK;
}

// The checks of a batch both step entry points share.  The reference's embedding lookup raises on an id outside the
// vocabulary.
int check_batch(const pllb_trainer_ctx* c, const char* who, const int32_t* ids, const int32_t* n_valid, int B, int T,
                int mode) {
  if (!ids || !n_valid || B < 1 || T < 1 || mode < 0 || mode > 2) return fail(PLLB_ERR_INVALID, std::string(who) + ": bad argument");
  if (T > c->t.max_seq)
    return fail(PLLB_ERR_TOO_LONG, "batch of " + std::to_string(T) + " positions; the trainer was created for " +
                                       std::to_string(c->t.max_seq));
  if ((int64_t)B * T > c->cap_rows)
    return fail(PLLB_ERR_OOM, "batch of " + std::to_string((int64_t)B * T) + " rows; the trainer was created for " +
                                  std::to_string(c->cap_rows));
  for (int i = 0; i < B * T; ++i)
    if (ids[i] < 0 || ids[i] >= c->d.vocab) return fail(PLLB_ERR_INVALID, "token id outside the vocabulary at row " + std::to_string(i));
  for (int b = 0; b < B; ++b)
    if (n_valid[b] < 1 || n_valid[b] > T) return fail(PLLB_ERR_INVALID, "n_valid must be in [1, T]");
  return PLLB_OK;
}

struct Upload { void* dst; const void* host; size_t bytes; };

// Host arrays -> device on s through the pinned staging buffer (packed back to back, one copy per array).
int upload(pllb_trainer_ctx* c, cudaStream_t s, std::initializer_list<Upload> arrays) {
  PLLB_CUDA(cudaStreamSynchronize(s));       // the pinned staging buffer of the previous call is free
  char* st = reinterpret_cast<char*>(c->host_stage);
  for (const Upload& a : arrays) {
    std::memcpy(st, a.host, a.bytes);
    PLLB_CUDA(cudaMemcpyAsync(a.dst, st, a.bytes, cudaMemcpyHostToDevice, s));
    st += a.bytes;
  }
  return PLLB_OK;
}

// operand copies and stash of the encoder layers, R rows
int alloc_enc_layers(pllb_trainer_ctx* c, int64_t R) {
  const int H = c->d.hidden, I = c->d.intermediate, NH = c->d.num_heads;
  const int64_t HH = (int64_t)H * H;
  for (auto& l : c->L) {
    RC(talloc(c, &l.qkv16, 3 * HH)); RC(talloc(c, &l.qkvT16, 3 * HH));
    RC(talloc(c, &l.ao16, HH)); RC(talloc(c, &l.aoT16, HH));
    RC(talloc(c, &l.ff116, (int64_t)I * H)); RC(talloc(c, &l.ff1T16, (int64_t)I * H));
    RC(talloc(c, &l.ff216, (int64_t)I * H)); RC(talloc(c, &l.ff2T16, (int64_t)I * H));
    RC(talloc(c, &l.x16, R * H)); RC(talloc(c, &l.qkv, R * 3 * H)); RC(talloc(c, &l.ctx, R * H));
    RC(talloc(c, &l.h1_16, R * H)); RC(talloc(c, &l.g16, R * I));
    RC(talloc(c, &l.lse, R * NH)); RC(talloc(c, &l.xhat1, R * H)); RC(talloc(c, &l.rstd1, R));
    RC(talloc(c, &l.f, R * I)); RC(talloc(c, &l.xhat2, R * H)); RC(talloc(c, &l.rstd2, R));
  }
  return PLLB_OK;
}

// The buffers every trainer has (R rows; `wide` = the widest GEMM output of a layer, Vw = the widest vocabulary-sized
// one, kmax = the widest GEMM input, stage_ints = int32 slots of the pinned upload buffer), the stream, the pinned
// buffers and the first operand refresh.  On failure the caller destroys the trainer.
int alloc_rest(pllb_trainer_ctx* c, int64_t R, int wide, int Vw, int kmax, int64_t stage_ints, const char* who) {
  const int H = c->d.hidden, NH = c->d.num_heads;
  const int64_t Rp = c->cap_rows_pad;
  RC(talloc(c, &c->ids, R)); RC(talloc(c, &c->n_valid, R));
  RC(talloc(c, &c->xhat_e, R * H)); RC(talloc(c, &c->rstd_e, R)); RC(talloc(c, &c->loss_dev, 2));
  RC(talloc(c, &c->h32, R * H)); RC(talloc(c, &c->y32, R * wide)); RC(talloc(c, &c->dh32, R * H));
  RC(talloc(c, &c->dz32, R * H)); RC(talloc(c, &c->dzd32, R * H)); RC(talloc(c, &c->Dq, R * NH));
  RC(talloc(c, &c->zeros, std::max(Vw, wide), true));
  RC(talloc(c, &c->colsum_scratch, (int64_t)2 * TRAIN_COLSUM_SPLITS * std::max(Vw, wide)));
  RC(talloc(c, &c->d16, R * std::max(wide, H))); RC(talloc(c, &c->dT16, (int64_t)std::max(wide, Vw) * Rp));
  RC(talloc(c, &c->xT16, (int64_t)kmax * Rp));
  RC(talloc(c, &c->params_dev, 1, true));
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    cudaGetLastError();
    return fail(PLLB_ERR_CUDA, std::string(who) + ": cudaStreamCreate failed");
  }
  if (const char* e = getenv("PLLB_TRAIN_GRAPH")) c->use_graph = atoi(e) != 0;
  if (cudaHostAlloc(&c->params_host, sizeof(TrainStepParams), cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&c->host_stage, sizeof(int32_t) * (size_t)stage_ints, cudaHostAllocDefault) != cudaSuccess) {
    cudaGetLastError();
    return fail(PLLB_ERR_OOM, std::string(who) + ": pinned staging buffer");
  }
  RC(refresh_all(c, 0));
  cudaError_t e = cudaStreamSynchronize(0);
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string(who) + ": " + cudaGetErrorString(e));
  return PLLB_OK;
}

// lin_w / lin_b / loss given: a RescoreBert (CLS) trainer; otherwise an MLM trainer (the head pointers of w are required)
int create_impl(pllb_trainer* out, const pllb_model_desc* desc, const pllb_weights* w, const pllb_train_desc* td, int device,
                const float* lin_w, const float* lin_b, const pllb_cls_loss_desc* loss) {
  const char* who = loss ? "pllb_cls_train_create" : "pllb_train_create";
  if (!out || !desc || !w || !w->layers || !td) return fail(PLLB_ERR_INVALID, std::string(who) + ": null argument");
  *out = nullptr;
  if (pllb_device_count() < 1) return fail(PLLB_ERR_NO_DEVICE, "no sm_100 (B200) device visible; libpllb200 has no CPU fallback");
  const pllb_model_desc& d = *desc;
  RC(check_model_shape(d));
  if (td->max_rows < 1 || td->max_seq < 1 || td->max_seq > d.max_position || td->max_seq > 512 ||
      td->hidden_dropout < 0.f || td->hidden_dropout >= 1.f || td->attention_dropout < 0.f || td->attention_dropout >= 1.f)
    return fail(PLLB_ERR_INVALID, std::string(who) + ": need max_rows >= 1, 1 <= max_seq <= min(max_position, 512), dropout in [0, 1)");
  if (loss && (!lin_w || !lin_b || !std::isfinite(loss->md_weight) || !std::isfinite(loss->mwer_weight) ||
               !std::isfinite(loss->am_weight) || loss->md_weight < 0.f || loss->mwer_weight < 0.f))
    return fail(PLLB_ERR_INVALID, "pllb_cls_train_create: need linear_w, linear_b and finite loss weights, md / mwer >= 0");
  PLLB_CUDA(cudaSetDevice(device));
  int major = 0;
  PLLB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(PLLB_ERR_NO_DEVICE, "device is not sm_100 (B200); libpllb200 has no other code path");
  pllb_trainer_ctx* c = new pllb_trainer_ctx();
  c->d = d;
  c->t = *td;
  c->device = device;
  c->cls = loss != nullptr;
  if (loss) c->loss = *loss;
  c->Vp = (int)round_up(d.vocab, 256);
  const int H = d.hidden, I = d.intermediate, V = d.vocab, NL = d.num_layers, Vp = c->Vp;
  const int64_t HH = (int64_t)H * H;
  int rc = PLLB_OK;
#define TRY(expr)                        \
  do {                                   \
    rc = (expr);                         \
    if (rc) { pllb_train_destroy(c); return rc; } \
  } while (0)
  // ---- flat layout
  int64_t cur = 0;
  c->word = take(cur, (int64_t)(c->cls ? V : Vp) * H);    // MLM: rows >= vocab stay zero (zero gradient, zero moments)
  c->pos = take(cur, (int64_t)d.max_position * H);
  c->type = take(cur, 2 * H);
  c->emb_g = take(cur, H);
  c->emb_b = take(cur, H);
  c->L.resize(NL);
  for (auto& l : c->L) {
    l.qkv_w = take(cur, 3 * HH); l.qkv_b = take(cur, 3 * H);
    l.ao_w = take(cur, HH); l.ao_b = take(cur, H); l.ao_g = take(cur, H); l.ao_be = take(cur, H);
    l.ff1_w = take(cur, (int64_t)I * H); l.ff1_b = take(cur, I);
    l.ff2_w = take(cur, (int64_t)H * I); l.ff2_b = take(cur, H); l.out_g = take(cur, H); l.out_be = take(cur, H);
  }
  if (c->cls) {
    c->lin_w = take(cur, H); c->lin_b = take(cur, 1);
  } else {
    c->head_w = take(cur, HH); c->head_b = take(cur, H); c->head_g = take(cur, H); c->head_be = take(cur, H);
    c->dec_b = take(cur, Vp);
  }
  c->n_flat = cur;
  TRY(talloc(c, &c->P, cur, true));
  TRY(talloc(c, &c->G, cur, true));
  TRY(talloc(c, &c->M, cur, true));
  TRY(talloc(c, &c->V, cur, true));
  // ---- parameters in
  TRY(visit_params(c, w, lin_w, lin_b,
                   [c](Span s, const float* src, int64_t n, int64_t off) { return copy_in(c, s, src, n, off); }));
  // ---- operand copies, stash, scratch
  c->cap_rows = td->max_rows;
  c->cap_rows_pad = round_up(c->cap_rows, 64);
  const int64_t R = c->cap_rows;
  const int wide = std::max(3 * H, I);
  TRY(alloc_enc_layers(c, R));
  // the MLM head's operand copies, stash, [R, Vp] logits and their gradient; a CLS trainer has none of them
  const int Vw = c->cls ? 0 : Vp;       // widest vocabulary-sized GEMM / column sum
  if (!c->cls) {
    TRY(talloc(c, &c->head16, HH)); TRY(talloc(c, &c->headT16, HH));
    TRY(talloc(c, &c->E16, (int64_t)Vp * H)); TRY(talloc(c, &c->ET16, (int64_t)Vp * H));
    TRY(talloc(c, &c->labels, R));
    TRY(talloc(c, &c->t_f32, R * H)); TRY(talloc(c, &c->xhat_h, R * H)); TRY(talloc(c, &c->rstd_h, R));
    TRY(talloc(c, &c->xlast16, R * H)); TRY(talloc(c, &c->tn16, R * H)); TRY(talloc(c, &c->dlogits16, R * Vp));
    TRY(talloc(c, &c->logits, R * Vp)); TRY(talloc(c, &c->loss_rows, R));
  } else {
    TRY(talloc(c, &c->group, R)); TRY(talloc(c, &c->target, R)); TRY(talloc(c, &c->am, R)); TRY(talloc(c, &c->err, R));
    TRY(talloc(c, &c->scores, R)); TRY(talloc(c, &c->dscore, R));
  }
  TRY(alloc_rest(c, R, wide, Vw, std::max(I, H), (c->cls ? 6 : 3) * R, who));
#undef TRY
  *out = c;
  return PLLB_OK;
}

// BART: the encoder layers above, the decoder layers, the stacked cross K / V and the LM head over shared
int create_s2s_impl(pllb_trainer* out, const pllb_s2s_desc* desc, const pllb_s2s_weights* w, const pllb_s2s_train_desc* td,
                    int device) {
  const char* who = "pllb_s2s_train_create";
  if (!out || !desc || !w || !w->enc.layers || !w->dec_layers || !td) return fail(PLLB_ERR_INVALID, std::string(who) + ": null argument");
  *out = nullptr;
  if (pllb_device_count() < 1) return fail(PLLB_ERR_NO_DEVICE, "no sm_100 (B200) device visible; libpllb200 has no CPU fallback");
  const pllb_s2s_desc& sd = *desc;
  const int H = sd.hidden, V = sd.vocab;
  if (H % 256 != 0 || H < 256 || H > 1024 || sd.num_heads * 64 != H || sd.enc_intermediate % 256 != 0 ||
      sd.dec_intermediate % 256 != 0 || sd.enc_intermediate < 256 || sd.dec_intermediate < 256 || sd.enc_layers < 1 ||
      sd.dec_layers < 1 || V < 1 || sd.enc_max_position < 1 || sd.dec_max_position < 1 || !std::isfinite(sd.embed_scale) ||
      !(sd.ln_eps > 0.f))
    return fail(PLLB_ERR_INVALID, std::string(who) + ": unsupported shape: need hidden in {256,512,768,1024}, head dim 64, "
                                                     "FFN widths % 256 == 0, >= 1 layer per stack");
  if (sd.operand_dtype != 0) return fail(PLLB_ERR_INVALID, std::string(who) + ": training takes operand_dtype 0 (bf16) only");
  if (td->max_batch < 1 || td->max_enc_len < 1 || td->max_dec_len < 1 || td->max_enc_len > std::min(sd.enc_max_position, 1024) ||
      td->max_dec_len > std::min(sd.dec_max_position, 1024) || !(td->dropout >= 0.f && td->dropout < 1.f) ||
      !(td->attention_dropout >= 0.f && td->attention_dropout < 1.f) || td->pad_id < 0 || td->pad_id >= V ||
      td->decoder_start_id < 0 || td->decoder_start_id >= V)
    return fail(PLLB_ERR_INVALID, std::string(who) + ": need capacities >= 1 with lengths <= min(max_position, 1024), "
                                                     "dropout in [0, 1), pad / decoder start ids in the vocabulary");
  PLLB_CUDA(cudaSetDevice(device));
  int major = 0;
  PLLB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(PLLB_ERR_NO_DEVICE, "device is not sm_100 (B200); libpllb200 has no other code path");
  pllb_trainer_ctx* c = new pllb_trainer_ctx();
  c->s2s = true;
  c->sd = sd;
  c->device = device;
  c->decoder_start_id = td->decoder_start_id;
  c->cap_batch = td->max_batch;
  c->cap_enc = td->max_enc_len;
  c->cap_dec = td->max_dec_len;
  // the shared encoder / optimizer code reads these two descriptors
  c->d = pllb_model_desc{sd.enc_layers, H, sd.num_heads, sd.enc_intermediate, V, sd.enc_max_position, sd.ln_eps,
                         sd.cls_id, sd.sep_id, 0, 0};
  c->t = pllb_train_desc{td->lr, td->beta1, td->beta2, td->adam_eps, td->weight_decay, td->dropout, td->attention_dropout,
                         td->seed, td->pad_id, 0, 0};
  c->Vp = (int)round_up(V, 256);
  const int NL = sd.dec_layers, Id = sd.dec_intermediate, Vp = c->Vp, NH = sd.num_heads;
  const int64_t HH = (int64_t)H * H;
  int rc = PLLB_OK;
#define TRY(expr)                        \
  do {                                   \
    rc = (expr);                         \
    if (rc) { pllb_train_destroy(c); return rc; } \
  } while (0)
  // ---- flat layout
  int64_t cur = 0;
  c->word = take(cur, (int64_t)Vp * H);            // shared; rows >= vocab stay zero
  c->pos = take(cur, (int64_t)(sd.enc_max_position + 2) * H);
  c->emb_g = take(cur, H);
  c->emb_b = take(cur, H);
  c->L.resize(sd.enc_layers);
  for (auto& l : c->L) {
    l.qkv_w = take(cur, 3 * HH); l.qkv_b = take(cur, 3 * H);
    l.ao_w = take(cur, HH); l.ao_b = take(cur, H); l.ao_g = take(cur, H); l.ao_be = take(cur, H);
    l.ff1_w = take(cur, (int64_t)sd.enc_intermediate * H); l.ff1_b = take(cur, sd.enc_intermediate);
    l.ff2_w = take(cur, (int64_t)H * sd.enc_intermediate); l.ff2_b = take(cur, H); l.out_g = take(cur, H); l.out_be = take(cur, H);
  }
  c->dec_pos = take(cur, (int64_t)(sd.dec_max_position + 2) * H);
  c->dec_emb_g = take(cur, H);
  c->dec_emb_b = take(cur, H);
  c->D.resize(NL);
  for (auto& l : c->D) {
    l.qkv_w = take(cur, 3 * HH); l.qkv_b = take(cur, 3 * H);
    l.o_w = take(cur, HH); l.o_b = take(cur, H); l.ln1_g = take(cur, H); l.ln1_b = take(cur, H);
    l.cq_w = take(cur, HH); l.cq_b = take(cur, H);
    l.co_w = take(cur, HH); l.co_b = take(cur, H); l.ln2_g = take(cur, H); l.ln2_b = take(cur, H);
    l.ff1_w = take(cur, (int64_t)Id * H); l.ff1_b = take(cur, Id);
    l.ff2_w = take(cur, (int64_t)H * Id); l.ff2_b = take(cur, H); l.ln3_g = take(cur, H); l.ln3_b = take(cur, H);
  }
  const int KV = 2 * H * NL;
  c->ckv_w = take(cur, (int64_t)KV * H);
  c->ckv_b = take(cur, KV);
  c->n_flat = cur;
  TRY(talloc(c, &c->P, cur, true));
  TRY(talloc(c, &c->G, cur, true));      // position rows 0 and 1 are never written: their gradient stays 0
  TRY(talloc(c, &c->M, cur, true));
  TRY(talloc(c, &c->V, cur, true));
  TRY(visit_s2s_params(c, w, [c](Span s, const float* src, int64_t n, int64_t off) { return copy_in(c, s, src, n, off); }));
  TRY(talloc(c, &c->flb, Vp, true));
  if (!w->final_logits_bias) TRY(fail(PLLB_ERR_INVALID, std::string(who) + ": final_logits_bias is null"));
  if (cudaMemcpyAsync(c->flb, w->final_logits_bias, sizeof(float) * V, cudaMemcpyDeviceToDevice, 0) != cudaSuccess) {
    cudaGetLastError();
    TRY(fail(PLLB_ERR_CUDA, std::string(who) + ": copy of final_logits_bias failed"));
  }
  // ---- operand copies, stash, scratch: the encoder and the decoder share row-sized buffers of max(T_enc, T_dec) rows
  c->cap_rows = (int64_t)td->max_batch * std::max(td->max_enc_len, td->max_dec_len);
  c->cap_rows_pad = round_up(c->cap_rows, 64);
  const int64_t R = c->cap_rows;
  TRY(alloc_enc_layers(c, R));
  for (auto& l : c->D) {
    TRY(talloc(c, &l.qkv16, 3 * HH)); TRY(talloc(c, &l.qkvT16, 3 * HH));
    TRY(talloc(c, &l.o16, HH)); TRY(talloc(c, &l.oT16, HH)); TRY(talloc(c, &l.cq16, HH)); TRY(talloc(c, &l.cqT16, HH));
    TRY(talloc(c, &l.co16, HH)); TRY(talloc(c, &l.coT16, HH));
    TRY(talloc(c, &l.ff116, (int64_t)Id * H)); TRY(talloc(c, &l.ff1T16, (int64_t)Id * H));
    TRY(talloc(c, &l.ff216, (int64_t)Id * H)); TRY(talloc(c, &l.ff2T16, (int64_t)Id * H));
    TRY(talloc(c, &l.x16, R * H)); TRY(talloc(c, &l.qkv, R * 3 * H)); TRY(talloc(c, &l.ctx, R * H));
    TRY(talloc(c, &l.h1_16, R * H)); TRY(talloc(c, &l.cq, R * H)); TRY(talloc(c, &l.cctx, R * H));
    TRY(talloc(c, &l.h2_16, R * H)); TRY(talloc(c, &l.g16, R * Id));
    TRY(talloc(c, &l.lse, R * NH)); TRY(talloc(c, &l.clse, R * NH));
    TRY(talloc(c, &l.xhat1, R * H)); TRY(talloc(c, &l.rstd1, R)); TRY(talloc(c, &l.xhat2, R * H)); TRY(talloc(c, &l.rstd2, R));
    TRY(talloc(c, &l.f, R * Id)); TRY(talloc(c, &l.xhat3, R * H)); TRY(talloc(c, &l.rstd3, R));
  }
  TRY(talloc(c, &c->ckv16, (int64_t)KV * H)); TRY(talloc(c, &c->ckvT16, (int64_t)KV * H));
  TRY(talloc(c, &c->E16, (int64_t)Vp * H)); TRY(talloc(c, &c->ET16, (int64_t)Vp * H));
  TRY(talloc(c, &c->labels, R)); TRY(talloc(c, &c->dec_ids, R));
  TRY(talloc(c, &c->xlast16, R * H)); TRY(talloc(c, &c->dlast16, R * H)); TRY(talloc(c, &c->ckv, R * KV));
  TRY(talloc(c, &c->dckv32, R * KV)); TRY(talloc(c, &c->dq32, R * H));
  TRY(talloc(c, &c->xhat_d, R * H)); TRY(talloc(c, &c->rstd_d, R));
  TRY(talloc(c, &c->dlogits16, R * Vp)); TRY(talloc(c, &c->logits, R * Vp)); TRY(talloc(c, &c->loss_rows, R));
  const int wide = std::max({3 * H, sd.enc_intermediate, Id, KV});
  TRY(alloc_rest(c, R, wide, Vp, std::max({sd.enc_intermediate, Id, H}), 4 * R, who));
#undef TRY
  *out = c;
  return PLLB_OK;
}

}  // namespace

extern "C" {

int pllb_train_create(pllb_trainer* out, const pllb_model_desc* desc, const pllb_weights* w, const pllb_train_desc* td,
                      int device) {
  return create_impl(out, desc, w, td, device, nullptr, nullptr, nullptr);
}

int pllb_train_destroy(pllb_trainer c) {
  if (!c) return PLLB_OK;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  for (auto& kv : c->graphs)
    if (kv.second.exec) cudaGraphExecDestroy(kv.second.exec);
  for (void* p : c->owned) cudaFree(p);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->host_stage) cudaFreeHost(c->host_stage);
  if (c->params_host) cudaFreeHost(c->params_host);
  delete c;
  return PLLB_OK;
}

int64_t pllb_train_workspace_bytes(pllb_trainer c) { return c ? c->owned_bytes : 0; }
int64_t pllb_train_kernel_launches(pllb_trainer c) { return c ? c->launches : 0; }
int64_t pllb_train_graph_replays(pllb_trainer c) { return c ? c->graph_replays : 0; }

int pllb_train_reset_optimizer(pllb_trainer c, float lr) {
  if (!c) return fail(PLLB_ERR_INVALID, "null trainer");
  PLLB_CUDA(cudaSetDevice(c->device));
  c->t.lr = lr;
  c->step = 0;
  PLLB_CUDA(cudaMemsetAsync(c->M, 0, sizeof(float) * (size_t)c->n_flat, c->stream));
  PLLB_CUDA(cudaMemsetAsync(c->V, 0, sizeof(float) * (size_t)c->n_flat, c->stream));
  return PLLB_OK;
}

int pllb_train_step_host(pllb_trainer c, const int32_t* input_ids, const int32_t* n_valid, const int32_t* labels, int32_t B,
                         int32_t T, int32_t mode, float* out_loss) {
  const char* who = "pllb_train_step_host";
  RC(require_kind(c, KIND_MLM, who));
  if (!labels) return fail(PLLB_ERR_INVALID, std::string(who) + ": bad argument");
  RC(check_batch(c, who, input_ids, n_valid, B, T, mode));
  const int R = B * T;
  for (int i = 0; i < R; ++i)      // the reference's CrossEntropyLoss raises on a label outside the vocabulary
    if (labels[i] < 0 || labels[i] >= c->d.vocab) return fail(PLLB_ERR_INVALID, "label outside the vocabulary at row " + std::to_string(i));
  PLLB_CUDA(cudaSetDevice(c->device));
  RC(upload(c, c->stream, {{c->ids, input_ids, sizeof(int32_t) * R}, {c->labels, labels, sizeof(int32_t) * R},
                           {c->n_valid, n_valid, sizeof(int32_t) * B}}));
  float loss = 0.f;
  RC(step_impl(c, B, T, mode, &loss, c->stream));
  c->last_rows = R;
  if (out_loss) *out_loss = loss;
  return PLLB_OK;
}

int pllb_train_row_losses_host(pllb_trainer c, float* out, int32_t n) {
  RC(require_kind(c, KIND_MLM, "pllb_train_row_losses_host", KIND_S2S));
  if (!out || n < 0 || n > c->last_rows) return fail(PLLB_ERR_INVALID, "pllb_train_row_losses_host: bad argument (n exceeds the rows of the last step)");
  PLLB_CUDA(cudaSetDevice(c->device));
  PLLB_CUDA(cudaMemcpyAsync(out, c->loss_rows, sizeof(float) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  PLLB_CUDA(cudaStreamSynchronize(c->stream));
  return PLLB_OK;
}

int pllb_train_export(pllb_trainer c, const pllb_weights* dst) {
  return export_params(c, false, false, dst, nullptr, nullptr, "pllb_train_export");
}

int pllb_train_export_grads(pllb_trainer c, const pllb_weights* dst) {
  return export_params(c, false, true, dst, nullptr, nullptr, "pllb_train_export_grads");
}

int pllb_cls_train_create(pllb_trainer* out, const pllb_model_desc* desc, const pllb_weights* w, const float* linear_w,
                          const float* linear_b, const pllb_train_desc* td, const pllb_cls_loss_desc* loss, int device) {
  if (!loss) return fail(PLLB_ERR_INVALID, "pllb_cls_train_create: null loss descriptor");
  return create_impl(out, desc, w, td, device, linear_w, linear_b, loss);
}

int pllb_cls_train_step_host(pllb_trainer c, const int32_t* input_ids, const int32_t* n_valid, const int32_t* group,
                             const float* target, const float* am, const float* err, int32_t B, int32_t T, int32_t mode,
                             float* out_loss, float* out_scores) {
  const char* who = "pllb_cls_train_step_host";
  RC(require_kind(c, KIND_CLS, who));
  if (!group || !target || !am || !err) return fail(PLLB_ERR_INVALID, std::string(who) + ": bad argument");
  RC(check_batch(c, who, input_ids, n_valid, B, T, mode));
  for (int b = 0; b < B; ++b) {
    if (b == 0 ? group[0] != 0 : (group[b] != group[b - 1] && group[b] != group[b - 1] + 1))
      return fail(PLLB_ERR_INVALID, "group must start at 0 and number the utterances in row order (each entry equal to the "
                                    "previous one or one more); bad entry at row " + std::to_string(b));
    if (!std::isfinite(target[b]) || !std::isfinite(am[b]) || !std::isfinite(err[b]))
      return fail(PLLB_ERR_INVALID, "non-finite target, AM score or error at row " + std::to_string(b));
  }
  PLLB_CUDA(cudaSetDevice(c->device));
  cudaStream_t s = c->stream;
  RC(upload(c, s, {{c->ids, input_ids, sizeof(int32_t) * B * T}, {c->n_valid, n_valid, sizeof(int32_t) * B},
                   {c->group, group, sizeof(int32_t) * B}, {c->target, target, sizeof(float) * B},
                   {c->am, am, sizeof(float) * B}, {c->err, err, sizeof(float) * B}}));
  float loss = 0.f;
  RC(step_impl(c, B, T, mode, &loss, s));
  if (out_scores) {
    PLLB_CUDA(cudaMemcpyAsync(out_scores, c->scores, sizeof(float) * B, cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaStreamSynchronize(s));
  }
  if (out_loss) *out_loss = loss;
  return PLLB_OK;
}

int pllb_cls_train_export(pllb_trainer c, const pllb_weights* dst, float* linear_w, float* linear_b) {
  return export_params(c, true, false, dst, linear_w, linear_b, "pllb_cls_train_export");
}

int pllb_cls_train_export_grads(pllb_trainer c, const pllb_weights* dst, float* linear_w, float* linear_b) {
  return export_params(c, true, true, dst, linear_w, linear_b, "pllb_cls_train_export_grads");
}

int pllb_s2s_train_create(pllb_trainer* out, const pllb_s2s_desc* desc, const pllb_s2s_weights* weights,
                          const pllb_s2s_train_desc* train, int device) {
  return create_s2s_impl(out, desc, weights, train, device);
}

int pllb_s2s_train_step_host(pllb_trainer c, const int32_t* input_ids, const int32_t* n_valid, const int32_t* labels,
                             int32_t B, int32_t T_enc, int32_t T_dec, int32_t mode, float* out_loss) {
  const char* who = "pllb_s2s_train_step_host";
  RC(require_kind(c, KIND_S2S, who));
  if (!input_ids || !n_valid || !labels || B < 1 || T_enc < 1 || T_dec < 1 || mode < 0 || mode > 2)
    return fail(PLLB_ERR_INVALID, std::string(who) + ": bad argument");
  if (T_enc > c->sd.enc_max_position || T_dec > c->sd.dec_max_position)
    return fail(PLLB_ERR_TOO_LONG, std::string(who) + ": T_enc " + std::to_string(T_enc) + " / T_dec " + std::to_string(T_dec) +
                                       " above the position tables (" + std::to_string(c->sd.enc_max_position) + " / " +
                                       std::to_string(c->sd.dec_max_position) + ")");
  if (B > c->cap_batch || T_enc > c->cap_enc || T_dec > c->cap_dec)
    return fail(PLLB_ERR_OOM, std::string(who) + ": batch [" + std::to_string(B) + ", " + std::to_string(T_enc) + ", " +
                                  std::to_string(T_dec) + "] above the capacity given at create [" + std::to_string(c->cap_batch) +
                                  ", " + std::to_string(c->cap_enc) + ", " + std::to_string(c->cap_dec) + "]");
  const int V = c->sd.vocab, Re = B * T_enc, Rd = B * T_dec;
  for (int i = 0; i < Re; ++i)
    if (input_ids[i] < 0 || input_ids[i] >= V) return fail(PLLB_ERR_INVALID, "token id outside the vocabulary at row " + std::to_string(i));
  for (int b = 0; b < B; ++b)
    if (n_valid[b] < 1 || n_valid[b] > T_enc) return fail(PLLB_ERR_INVALID, "n_valid must be in [1, T_enc]");
  int n_lab = 0;
  for (int i = 0; i < Rd; ++i) {
    if (labels[i] == -100) continue;
    if (labels[i] < 0 || labels[i] >= V)
      return fail(PLLB_ERR_INVALID, "label outside the vocabulary (and not -100) at position " + std::to_string(i));
    ++n_lab;
  }
  if (n_lab == 0) return fail(PLLB_ERR_INVALID, std::string(who) + ": every label is -100 (the mean loss is undefined)");
  // decoder input = shift_tokens_right(labels, pad_id, decoder_start_id)
  c->dec_host.resize(Rd);
  for (int b = 0; b < B; ++b) {
    c->dec_host[(size_t)b * T_dec] = c->decoder_start_id;
    for (int t = 1; t < T_dec; ++t) {
      const int32_t l = labels[(size_t)b * T_dec + t - 1];
      c->dec_host[(size_t)b * T_dec + t] = l == -100 ? c->t.pad_id : l;
    }
  }
  PLLB_CUDA(cudaSetDevice(c->device));
  RC(upload(c, c->stream, {{c->ids, input_ids, sizeof(int32_t) * Re}, {c->n_valid, n_valid, sizeof(int32_t) * B},
                           {c->labels, labels, sizeof(int32_t) * Rd}, {c->dec_ids, c->dec_host.data(), sizeof(int32_t) * Rd}}));
  float loss = 0.f;
  RC(step_impl(c, B, T_enc, mode, &loss, c->stream, T_dec));
  c->last_rows = Rd;
  if (out_loss) *out_loss = loss;
  return PLLB_OK;
}

namespace {
int export_s2s(pllb_trainer c, bool grads, const pllb_s2s_weights* w, const char* who) {
  RC(require_kind(c, KIND_S2S, who));
  if (!w || !w->enc.layers || !w->dec_layers) return fail(PLLB_ERR_INVALID, std::string(who) + ": null argument");
  const float* buf = grads ? c->G : c->P;
  PLLB_CUDA(cudaSetDevice(c->device));
  PLLB_CUDA(cudaStreamSynchronize(c->stream));
  RC(visit_s2s_params(c, w, [buf](Span s, const float* dst, int64_t n, int64_t off) { return copy_out(buf, s, dst, n, off); }));
  if (w->final_logits_bias) {       // a buffer: the given values, no gradient
    float* dst = const_cast<float*>(w->final_logits_bias);
    if (grads) PLLB_CUDA(cudaMemsetAsync(dst, 0, sizeof(float) * c->sd.vocab, 0));
    else PLLB_CUDA(cudaMemcpyAsync(dst, c->flb, sizeof(float) * c->sd.vocab, cudaMemcpyDeviceToDevice, 0));
  }
  PLLB_CUDA(cudaStreamSynchronize(0));
  return PLLB_OK;
}
}  // namespace

int pllb_s2s_train_export(pllb_trainer c, const pllb_s2s_weights* dst) {
  return export_s2s(c, false, dst, "pllb_s2s_train_export");
}

int pllb_s2s_train_export_grads(pllb_trainer c, const pllb_s2s_weights* dst) {
  return export_s2s(c, true, dst, "pllb_s2s_train_export_grads");
}

// ---------------------------------------------------------------- kernel test hooks (pllb_debug_train_*)
// Thin wrappers over the launchers of train.h on caller buffers, so each kernel can be checked alone against a
// high-precision reference.  Scalars and pointers are checked first; then the DEVICE index arrays a kernel reads
// without bounds (n_valid, ids, labels) are copied back and checked, so a bad argument never reaches a launch.
namespace {
bool hidden_ok(int H) { return H == 256 || H == 512 || H == 768 || H == 1024; }

int bad(const char* who, const std::string& what) { return fail(PLLB_ERR_INVALID, std::string(who) + ": " + what); }

int need_device(const char* who) {
  if (pllb_device_count() < 1) return fail(PLLB_ERR_NO_DEVICE, std::string(who) + ": no sm_100 (B200) device visible");
  return PLLB_OK;
}

// every entry of the DEVICE int32[n] in [lo, hi], or equal to `also` (when also_ok)
int check_dev_ints(const char* who, const char* name, const int32_t* d, int64_t n, int lo, int hi, cudaStream_t s,
                   bool also_ok = false, int also = 0, int* count_also = nullptr) {
  std::vector<int32_t> h((size_t)n);
  PLLB_CUDA(cudaMemcpyAsync(h.data(), d, sizeof(int32_t) * (size_t)n, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  int k = 0;
  for (int64_t i = 0; i < n; ++i) {
    if (also_ok && h[i] == also) { ++k; continue; }
    if (h[i] < lo || h[i] > hi)
      return bad(who, std::string(name) + "[" + std::to_string(i) + "] = " + std::to_string(h[i]) + " outside [" +
                          std::to_string(lo) + ", " + std::to_string(hi) + "]");
  }
  if (count_also) *count_also = k;
  return PLLB_OK;
}

bool drop_ok(const uint64_t* seed, float p) { return p >= 0.f && p < 1.f && (p == 0.f || seed); }

// the attention kernels read bf16 rows and the fp32 dctx 16 bytes at a time and write the fp32 gradients as pairs
bool aligned(const void* p, uintptr_t bytes) { return p == nullptr || reinterpret_cast<uintptr_t>(p) % bytes == 0; }
}  // namespace

int pllb_debug_train_attn(const uint16_t* qkv, const int32_t* n_valid, int32_t B, int32_t T, int32_t H, const float* dctx,
                          const uint64_t* seed, float p, uint32_t site, uint16_t* ctx, float* lse, float* dqkv, float* Dscratch,
                          void* stream) {
  const char* who = "pllb_debug_train_attn";
  if (!qkv || !n_valid || !ctx || !lse) return bad(who, "null pointer");
  if (dctx && (!dqkv || !Dscratch)) return bad(who, "the backward pass needs dqkv and Dscratch");
  if (B < 1 || T < 1 || T > 512) return bad(who, "need B >= 1 and T in [1, 512]");
  if (!hidden_ok(H)) return bad(who, "hidden must be 256, 512, 768 or 1024");
  if (!drop_ok(seed, p)) return bad(who, "need p in [0, 1) and a seed when p > 0");
  if (!aligned(qkv, 16) || !aligned(dctx, 16) || !aligned(ctx, 4) || !aligned(lse, 4) || !aligned(dqkv, 8) ||
      !aligned(Dscratch, 4))
    return bad(who, "misaligned pointer (qkv and dctx: 16 bytes, dqkv: 8, ctx, lse and Dscratch: 4)");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  RC(check_dev_ints(who, "n_valid", n_valid, B, 1, T, s));
  const TrainDrop d = drop_of(seed, p);
  const int R = B * T, NH = H / 64;
  RC(launch_train_attn_fwd(qkv, n_valid, R, T, H, NH, d, site, ctx, lse, s));
  if (dctx) RC(launch_train_attn_bwd(qkv, dctx, lse, n_valid, R, T, H, NH, d, site, dqkv, Dscratch, s));
  return PLLB_OK;
}

int pllb_debug_s2s_attn(const uint16_t* q, const uint16_t* k, const uint16_t* v, int32_t ldq, int32_t ldkv,
                        const int32_t* n_valid, int32_t B, int32_t Tq, int32_t Tk, int32_t NH, int32_t causal,
                        const float* dctx, const uint64_t* seed, float p, uint32_t site, uint16_t* ctx, float* lse, float* dq,
                        int32_t lddq, float* dk, float* dv, int32_t lddkv, float* Dscratch, void* stream) {
  const char* who = "pllb_debug_s2s_attn";
  if (!q || !k || !v || !ctx || !lse || (!causal && !n_valid)) return bad(who, "null pointer");
  if (dctx && (!dq || !dk || !dv || !Dscratch)) return bad(who, "the backward pass needs dq, dk, dv and Dscratch");
  if (B < 1 || Tq < 1 || Tq > 512 || Tk < 1 || Tk > 512 || (causal && Tq != Tk))
    return bad(who, "need B >= 1, Tq and Tk in [1, 512], Tq == Tk when causal");
  const int H = NH * 64;
  if (NH < 1 || !hidden_ok(H)) return bad(who, "NH * 64 must be 256, 512, 768 or 1024");
  // 16-byte rows for the vector loads of Q, K and V (the dk / dv pass reads Q rows as K rows are read), 8-byte rows
  // (fp32 pairs) for the gradients
  if (ldq < H || ldkv < H || ldq % 8 || ldkv % 8 || (dctx && (lddq < H || lddkv < H || lddq % 2 || lddkv % 2)))
    return bad(who, "bad row stride");
  if (!drop_ok(seed, p)) return bad(who, "need p in [0, 1) and a seed when p > 0");
  if (!aligned(q, 16) || !aligned(k, 16) || !aligned(v, 16) || !aligned(dctx, 16) || !aligned(ctx, 4) ||
      !aligned(lse, 4) || !aligned(dq, 8) || !aligned(dk, 8) || !aligned(dv, 8) || !aligned(Dscratch, 4))
    return bad(who, "misaligned pointer (q, k, v and dctx: 16 bytes, dq, dk and dv: 8, ctx, lse and Dscratch: 4)");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  if (!causal) RC(check_dev_ints(who, "n_valid", n_valid, B, 1, Tk, s));
  const S2sAttn a{q, k, v, ldq, ldkv, B, Tq, Tk, NH, causal != 0, causal ? nullptr : n_valid};
  const TrainDrop d = drop_of(seed, p);
  RC(launch_train_attn_s2s_fwd(a, d, site, ctx, lse, s));
  if (dctx) RC(launch_train_attn_s2s_bwd(a, dctx, lse, d, site, dq, lddq, dk, dv, lddkv, Dscratch, s));
  return PLLB_OK;
}

int pllb_debug_train_ln_fwd(int32_t form, const float* y, const float* res, const int32_t* ids, int32_t T, const float* word,
                            int32_t vocab, const float* pos, const float* type, float embed_scale, const float* g, const float* b,
                            float eps, int32_t R, int32_t H, const uint64_t* seed, float p, uint32_t site, float* out32,
                            uint16_t* out16, float* xhat, float* rstd, void* stream) {
  const char* who = "pllb_debug_train_ln_fwd";
  if (form < 0 || form > 2) return bad(who, "form must be 0 (plain), 1 (BERT embedding) or 2 (BART embedding)");
  if (!g || !b || (form == 0 && !y) || (form != 0 && (!ids || !word || !pos || (form == 1 && !type))) ||
      (form == 2 && (!out32 || !out16 || !xhat || !rstd)))
    return bad(who, "null pointer");
  if (R < 1 || !(eps > 0.f)) return bad(who, "need R >= 1 and eps > 0");
  if (form != 0 && (T < 1 || T > 512 || vocab < 1)) return bad(who, "need T in [1, 512] and vocab >= 1");
  if (!hidden_ok(H)) return bad(who, "hidden must be 256, 512, 768 or 1024");
  if (!drop_ok(seed, p)) return bad(who, "need p in [0, 1) and a seed when p > 0");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  if (form != 0) RC(check_dev_ints(who, "ids", ids, R, 0, vocab - 1, s));
  const TrainDrop d = drop_of(seed, p);
  if (form == 0) return launch_train_ln_fwd(y, res, g, b, eps, R, H, d, site, out32, out16, xhat, rstd, s);
  if (form == 1) return launch_train_embed(ids, T, word, pos, type, g, b, eps, R, H, d, site, out32, out16, xhat, rstd, s);
  return launch_train_bart_embed(ids, T, word, embed_scale, pos, g, b, eps, R, H, d, site, out32, out16, xhat, rstd, s);
}

int pllb_debug_train_ln_bwd(float* dy, const float* add, const float* g, const float* xhat, const float* rstd, int32_t R,
                            int32_t H, const uint64_t* seed, float p, int32_t site_in, int32_t site_out, float* dz,
                            float* dz_drop, void* stream) {
  const char* who = "pllb_debug_train_ln_bwd";
  if (!dy || !g || !xhat || !rstd || !dz) return bad(who, "null pointer");
  if (R < 1) return bad(who, "need R >= 1");
  if (!hidden_ok(H)) return bad(who, "hidden must be 256, 512, 768 or 1024");
  if (!drop_ok(seed, p) || site_in < -1 || site_out < -1) return bad(who, "need p in [0, 1), a seed when p > 0, sites >= -1");
  RC(need_device(who));
  return launch_train_ln_bwd(dy, add, g, xhat, rstd, R, H, drop_of(seed, p), site_in, site_out, dz, dz_drop,
                             (cudaStream_t)stream);
}

int pllb_debug_train_ce(const float* logits, const int32_t* labels, int32_t R, int32_t V, int32_t Vp, int32_t ignore_index,
                        float* loss_rows, uint16_t* dlogits, float* out_loss, void* stream) {
  const char* who = "pllb_debug_train_ce";
  if (!logits || !labels || !loss_rows || !out_loss) return bad(who, "null pointer");
  if (R < 1 || V < 1 || Vp < V) return bad(who, "need R >= 1 and 1 <= V <= Vp");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  if (!ignore_index) {
    RC(check_dev_ints(who, "labels", labels, R, 0, V - 1, s));
    return launch_train_ce(logits, labels, R, V, Vp, loss_rows, dlogits, out_loss, s);
  }
  int ignored = 0;
  RC(check_dev_ints(who, "labels", labels, R, 0, V - 1, s, true, -100, &ignored));
  if (ignored == R) return bad(who, "every label is -100");
  return launch_train_ce_ignore(logits, labels, R, V, Vp, loss_rows, dlogits, out_loss, s);
}

int pllb_debug_train_embed_bwd(int32_t form, float* dz, const int32_t* ids, int32_t B, int32_t T, int32_t H, int32_t pos_rows,
                               int32_t pad_id, float scale, float* dword, int32_t vocab, float* dpos, float* dtype0,
                               float* scratch, void* stream) {
  const char* who = "pllb_debug_train_embed_bwd";
  if (form < 0 || form > 1) return bad(who, "form must be 0 (BERT embedding) or 1 (BART embedding)");
  if (!dz || !ids || !dword || !dpos || (form == 0 && !dtype0)) return bad(who, "null pointer");
  if (B < 1 || T < 1 || T > 512 || pos_rows < T || vocab < 1) return bad(who, "need B >= 1, T in [1, 512], pos_rows >= T");
  if (!hidden_ok(H)) return bad(who, "hidden must be 256, 512, 768 or 1024");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  RC(check_dev_ints(who, "ids", ids, (int64_t)B * T, 0, vocab - 1, s));
  if (form == 0) return launch_train_embed_bwd(dz, ids, B, T, H, pos_rows, pad_id, dword, dpos, dtype0, scratch, s);
  return launch_train_bart_embed_bwd(dz, ids, B, T, H, pos_rows, pad_id, scale, dword, dpos, s);
}

int pllb_debug_train_colsum(const void* dy, int32_t dy_bf16, const float* xhat, int32_t R, int32_t C, float* out_sum,
                            float* out_dot, float* scratch, void* stream) {
  const char* who = "pllb_debug_train_colsum";
  if (!dy || (!out_sum && !out_dot) || (out_dot && !xhat)) return bad(who, "null pointer");
  if (R < 1 || C < 1) return bad(who, "need R >= 1 and C >= 1");
  RC(need_device(who));
  return launch_train_colsum(dy, dy_bf16 != 0, xhat, R, C, out_sum, out_dot, scratch, (cudaStream_t)stream);
}

int pllb_debug_train_cast_transpose(const void* src, int32_t src_bf16, int32_t R, int32_t C, int32_t Rp, uint16_t* dst16,
                                    uint16_t* dstT, void* stream) {
  const char* who = "pllb_debug_train_cast_transpose";
  if (!src || (!dst16 && !dstT)) return bad(who, "null pointer");
  if (R < 1 || C < 1 || Rp < R) return bad(who, "need R >= 1, C >= 1 and Rp >= R");
  RC(need_device(who));
  return launch_train_cast_transpose(src, src_bf16 != 0, R, C, Rp, dst16, dstT, (cudaStream_t)stream);
}

int pllb_debug_train_gelu(const float* f, int64_t n, uint16_t* out16, float* out32, float* dg, void* stream) {
  const char* who = "pllb_debug_train_gelu";
  if (!f || (!out16 && !out32 && !dg)) return bad(who, "null pointer");
  if (n < 1) return bad(who, "need n >= 1");
  RC(need_device(who));
  cudaStream_t s = (cudaStream_t)stream;
  if (out16 || out32) RC(launch_train_gelu_fwd(f, n, out16, out32, s));
  if (dg) RC(launch_train_gelu_bwd(dg, f, n, s));
  return PLLB_OK;
}

}  // extern "C"
