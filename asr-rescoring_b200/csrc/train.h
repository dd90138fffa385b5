// train.h — launchers of train_kernels.cu (MLM fine-tuning path; see train_api.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pllb {

// Scalars that change from step to step live in DEVICE memory (written before every step), not in
// kernel arguments, so a captured CUDA graph of the step can be replayed unchanged.
struct TrainStepParams {
  uint64_t seed;          // dropout: run seed mixed with the forward-pass number
  float adam_step_size;   // lr / (1 - beta1^t)
  float adam_bc2_sqrt;    // sqrt(1 - beta2^t)
};

struct TrainDrop {        // stateless dropout (train_kernels.cu: drop_factor)
  const uint64_t* seed;   // DEVICE pointer (TrainStepParams.seed)
  uint32_t thresh;        // drop iff hash < thresh; 0 = no dropout
  float inv_keep;         // 1 / (1 - p)
};

// out = [dropout](LN(word[ids] + pos[r % T] + type[0]))   (BertEmbeddings); fp32 + bf16 copies, saved xhat / rstd
int launch_train_embed(const int32_t* ids, int T, const float* word, const float* pos, const float* type, const float* g,
                       const float* b, float eps, int R, int H, TrainDrop drop, uint32_t site, float* out32, void* out16,
                       float* xhat, float* rstd, cudaStream_t s);
// out = LN(dropout(y) + res)   (BertSelfOutput / BertOutput; res == nullptr: the head's transform LayerNorm)
int launch_train_ln_fwd(const float* y, const float* res, const float* g, const float* b, float eps, int R, int H,
                        TrainDrop drop, uint32_t site, float* out32, void* out16, float* xhat, float* rstd, cudaStream_t s);
// dy <- (dy + add) [* dropout mask site_in]; dz = LayerNorm backward; dz_drop = dz [* dropout mask site_out]
int launch_train_ln_bwd(float* dy, const float* add, const float* g, const float* xhat, const float* rstd, int R, int H,
                        TrainDrop drop, int site_in, int site_out, float* dz, float* dz_drop, cudaStream_t s);
// out_sum[c] = sum_r dy[r,c]; out_dot[c] = sum_r dy[r,c] * xhat[r,c] (either may be null).
// scratch: 2 * TRAIN_COLSUM_SPLITS * C floats for the row-sliced form (nullptr: one slice)
constexpr int TRAIN_COLSUM_SPLITS = 64;
int launch_train_colsum(const void* dy, bool dy_bf16, const float* xhat, int R, int C, float* out_sum, float* out_dot,
                        float* scratch, cudaStream_t s);
int launch_train_gelu_fwd(const float* f, int64_t n, void* out16, float* out32, cudaStream_t s);
int launch_train_gelu_bwd(float* dg, const float* f, int64_t n, cudaStream_t s);
// src [R, C] (fp32 or bf16) -> dst16 [R, C] and / or dstT [C, Rp] (bf16; transposed columns >= R zero)
int launch_train_cast_transpose(const void* src, bool src_bf16, int R, int C, int Rp, void* dst16, void* dstT,
                                cudaStream_t s);
int launch_train_attn_fwd(const void* qkv, const int32_t* n_valid, int R, int T, int H, int NH, TrainDrop drop, uint32_t site,
                          void* ctx, float* lse, cudaStream_t s);
int launch_train_attn_bwd(const void* qkv, const float* dctx, const float* lse, const int32_t* n_valid, int R, int T, int H,
                          int NH, TrainDrop drop, uint32_t site, float* dqkv, float* Dscratch, cudaStream_t s);
int launch_train_scale(float* x, int64_t n, float alpha, cudaStream_t s);
// per-row cross entropy over V of the Vp logit columns, mean loss, dlogits = softmax - onehot (bf16, may be null;
// the 1/R of the mean is applied by the caller in fp32)
int launch_train_ce(const float* logits, const int32_t* labels, int R, int V, int Vp, float* loss_rows, void* dlogits,
                    float* out_loss, cudaStream_t s);
int launch_train_embed_bwd(const float* dz, const int32_t* ids, int B, int T, int H, int max_pos, int pad_id, float* dword,
                           float* dpos, float* dtype0, float* scratch, cudaStream_t s);
// scalars: DEVICE TrainStepParams (adam_step_size, adam_bc2_sqrt of this step)
int launch_train_adamw(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                       float wd, const TrainStepParams* scalars, cudaStream_t s);

// RescoreBert head (pllb_cls_train_*): scores[b] = w . h[b*T, :] + b[0] over the fp32 last-layer output h [B*T, H]
int launch_train_cls_fwd(const float* h, const float* w, const float* b, int B, int T, int H, float* scores, cudaStream_t s);
// MD + MWER loss of the B scores (group: DEVICE int32[B], 0-based and contiguous); dscore may be null (no backward)
int launch_train_cls_loss(const float* scores, const float* target, const float* am, const float* err, const int32_t* group,
                          int B, float md_weight, float mwer_weight, float am_weight, float* dscore, float* out_loss,
                          cudaStream_t s);
// dw [H], db [1]: head gradients; dh [B*T, H]: the top-layer gradient the encoder backward starts from
int launch_train_cls_bwd(const float* h, const float* w, const float* dscore, int B, int T, int H, float* dw, float* db,
                         float* dh, cudaStream_t s);

// ---- BART fine-tuning (pllb_s2s_train_*)
// out = [dropout](LN(word[ids] * scale + pos[r % T]))   (BART embeddings; pos = row 2 of embed_positions)
int launch_train_bart_embed(const int32_t* ids, int T, const float* word, float scale, const float* pos, const float* g,
                            const float* b, float eps, int R, int H, TrainDrop drop, uint32_t site, float* out32, void* out16,
                            float* xhat, float* rstd, cudaStream_t s);
// dpos[p] = sum_b dz[b*T + p] for p < pos_rows (0 past T); then dz *= scale (in place) and dword[id] += the
// occurrences of id, pad_id excluded
int launch_train_bart_embed_bwd(float* dz, const int32_t* ids, int B, int T, int H, int pos_rows, int pad_id, float scale,
                                float* dword, float* dpos, cudaStream_t s);
// One attention of B sequences: Tq bf16 query rows (q, row stride ldq) over Tk key / value rows (k, v, stride ldkv),
// head h at columns h*64.  causal: Tq == Tk, query i sees keys <= i; otherwise keys < n_valid[seq] (DEVICE int32[B]).
struct S2sAttn {
  const void *q, *k, *v;
  int ldq, ldkv;
  int B, Tq, Tk, NH;
  bool causal;
  const int32_t* n_valid;
};
// ctx bf16 [B*Tq, NH*64], lse [B*Tq*NH]
int launch_train_attn_s2s_fwd(const S2sAttn& a, TrainDrop drop, uint32_t site, void* ctx, float* lse, cudaStream_t s);
// dq fp32 (row stride lddq), dk / dv fp32 (row stride lddkv); Dscratch [B*Tq*NH]
int launch_train_attn_s2s_bwd(const S2sAttn& a, const float* dctx, const float* lse, TrainDrop drop, uint32_t site, float* dq,
                              int lddq, float* dk, float* dv, int lddkv, float* Dscratch, cudaStream_t s);
// cross entropy with ignore_index -100 (loss 0, zero dlogits row); out_loss2[0] = mean over the N labelled rows,
// out_loss2[1] = 1 / N (fp32, DEVICE: read by launch_train_scale_dev)
int launch_train_ce_ignore(const float* logits, const int32_t* labels, int R, int V, int Vp, float* loss_rows, void* dlogits,
                           float* out_loss2, cudaStream_t s);
int launch_train_scale_dev(float* x, int64_t n, const float* alpha, cudaStream_t s);

}  // namespace pllb
