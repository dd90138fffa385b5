/*
 * pllb.h — C ABI of libpllb200.so, the B200-native MLM-PLL N-best scoring path.
 *
 * The reference (ishine/ASR-Rescoring) is pure Python and has no FFI for this
 * path; the boundary that exists is a set of Python functions.  Each entry
 * point below names the reference interface it replaces (file:line relative to
 * the reference tree).  INTEGRATION.md shows the ctypes binding a maintainer of
 * the reference would add.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns 0 on success or a
 *     non-zero pllb_status, and pllb_last_error() gives the message.
 *   - "_host" entry points take HOST buffers and do their own H2D/D2H copies
 *     (this is what the end-to-end benchmark times).  The others take DEVICE
 *     pointers owned by the caller (torch allocations) plus a cudaStream_t
 *     passed as void*; they never synchronise the device unless stated.
 *   - one handle per GPU, driven from one host thread.  There is no CPU
 *     fallback: without a usable sm_100 device every compute call fails.
 */
#ifndef PLLB_H_
#define PLLB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PLLB_ABI_VERSION 1

typedef enum pllb_status {
  PLLB_OK = 0,
  PLLB_ERR_INVALID = 1,     /* bad argument / unsupported model shape          */
  PLLB_ERR_CUDA = 2,        /* CUDA runtime / driver error                      */
  PLLB_ERR_NO_DEVICE = 3,   /* no sm_100 GPU visible (there is no CPU fallback) */
  PLLB_ERR_OOM = 4,         /* workspace does not fit                           */
  PLLB_ERR_TOO_LONG = 5     /* a hypothesis exceeds max_position_embeddings-2   */
} pllb_status;

typedef struct pllb_context* pllb_handle;

/* Model shape.  Mirrors transformers.BertConfig as used by
 * MLM_PLL/main.py:184 (BertForMaskedLM.from_pretrained(config.model.bert)). */
typedef struct pllb_model_desc {
  int32_t num_layers;     /* 12 (bert-base-chinese) / 24                     */
  int32_t hidden;         /* 768 / 1024; multiple of 256                     */
  int32_t num_heads;      /* hidden / 64 (head dim is fixed at 64)           */
  int32_t intermediate;   /* 3072 / 4096; multiple of 256                    */
  int32_t vocab;          /* 21128                                           */
  int32_t max_position;   /* 512                                             */
  float   ln_eps;         /* 1e-12                                           */
  int32_t cls_id, sep_id, mask_id; /* 101, 102, 103                          */
  int32_t operand_dtype;  /* GEMM / attention operand type, fp32 accumulate
                             in every mode:
                             0 = bf16 activations and weights;
                             1 = IEEE fp16 activations and weights (same
                                 tensor-core rate, 3 more mantissa bits: ~8x
                                 smaller PLL error; conversions saturate at
                                 +-65504 instead of overflowing);
                             2 = bf16 encoder, fp16 MLM head (transform +
                                 decoder operands; 1 % of the FLOPs, removes
                                 the largest single rounding site);
                             3 = bf16 for encoder layers < NL/2, fp16 for the
                                 layers >= NL/2 and the head;
                             16 + k = bf16 for layers < k, fp16 from layer k on
                                 and in the head (16 = mode 1, 16 + NL = mode 2) */
} pllb_model_desc;

/* One encoder layer; DEVICE pointers to fp32 tensors in nn.Linear layout
 * ([out_features, in_features] row-major), i.e. the tensors of the
 * BertForMaskedLM state_dict loaded at MLM_PLL/main.py:185-187. */
typedef struct pllb_layer_weights {
  const float *q_w, *q_b, *k_w, *k_b, *v_w, *v_b;   /* attention.self.{query,key,value} */
  const float *ao_w, *ao_b, *ao_ln_g, *ao_ln_b;     /* attention.output.{dense,LayerNorm} */
  const float *ff1_w, *ff1_b;                       /* intermediate.dense  */
  const float *ff2_w, *ff2_b, *out_ln_g, *out_ln_b; /* output.{dense,LayerNorm} */
} pllb_layer_weights;

typedef struct pllb_weights {
  const float *word_emb, *pos_emb, *type_emb, *emb_ln_g, *emb_ln_b; /* bert.embeddings.* */
  const pllb_layer_weights* layers;  /* HOST array of num_layers structs */
  const float *head_w, *head_b, *head_ln_g, *head_ln_b; /* cls.predictions.transform.* */
  const float *decoder_w;   /* cls.predictions.decoder.weight [vocab, hidden] (tied to word_emb) */
  const float *decoder_b;   /* cls.predictions.bias [vocab] */
} pllb_weights;

/* Counters filled by pllb_get_stats (since create or the last reset). */
typedef struct pllb_stats {
  int64_t kernel_launches;   /* kernels of this library launched            */
  int64_t hyps_scored, copies_scored, tokens_expanded;
  int64_t chunks;
  double  gemm_flops;        /* algorithmic FLOPs issued to the GEMM kernel */
  float   last_gemm_ms;      /* device time of the GEMM kernels of the last
                                pllb_score call when timing is enabled      */
  float   last_total_ms;     /* device time of the last pllb_score call     */
  int64_t last_gemm_launches;
} pllb_stats;

const char* pllb_last_error(void);
int pllb_abi_version(void);

/* Number of CUDA devices usable by this library (compute capability 10.x).
 * Returns 0 when none: callers must fail, there is no fallback. */
int pllb_device_count(void);

/* ---- PLL scoring: replaces MLM_PLL/main.py:73-114 (run_one_epoch, scoring
 * branch), :28-54 (collate) and MLM_PLL/preprocess.py:9-30 (masked-copy
 * expansion).  Weights are converted to bf16 GEMM operands once here.
 * max_chunk_tokens bounds the expanded tokens (sum over hyps of L*(L+2))
 * processed per internal chunk and therefore the workspace size; 0 = default. */
int pllb_create(pllb_handle* out, const pllb_model_desc* desc,
                const pllb_weights* weights, int64_t max_chunk_tokens, int device);
int pllb_destroy(pllb_handle h);

/* Bytes of device workspace owned by the handle. */
int64_t pllb_workspace_bytes(pllb_handle h);

/* hyp_tokens   DEVICE int32[hyp_offsets[n_hyp]]  wordpiece ids, no specials; hypothesis i
 *                                                is hyp_tokens[hyp_offsets[i] .. hyp_offsets[i+1])
 * hyp_offsets  HOST   int64[n_hyp+1]             (control metadata)
 * out_pll      DEVICE double[n_hyp]   sum over the L masked copies of
 *                                     log_softmax(logits[mask_pos])[token]
 *                                     (a hypothesis with L == 0 gets 0.0)
 * out_token_logp DEVICE float[hyp_offsets[n_hyp]] or NULL; the individual terms
 * Asynchronous on `stream`: hyp_offsets is consumed before the call returns, the
 * device buffers when the stream reaches the work.  A handle owns ONE workspace:
 * use it from one host thread and issue its calls on one stream (calls may be queued
 * back to back without synchronising; work on different streams must be ordered by
 * the caller). */
int pllb_score(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
               int32_t n_hyp, double* out_pll, float* out_token_logp, void* stream);

/* Same with HOST buffers; copies in, scores, copies out, synchronises. */
int pllb_score_host(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
                    int32_t n_hyp, double* out_pll, float* out_token_logp);

/* ---- Sequence-level scoring: replaces the forward of RescoreBert/model.py:13-21 inside
 * RescoreBert/main.py run_one_epoch (scoring, :232-285): every hypothesis goes through the
 * encoder ONCE as [CLS] t [SEP] and out[i] = dot(last_hidden_state[i, 0, :], linear_w) +
 * linear_b.  The handle may be created without MLM head weights (head_w == NULL ...).
 * linear_w DEVICE float[hidden] (HOST in the _host variant); out_scores float[n_hyp]. */
int pllb_score_cls(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
                   int32_t n_hyp, const float* linear_w, float linear_b, float* out_scores,
                   void* stream);
int pllb_score_cls_host(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
                        int32_t n_hyp, const float* linear_w, float linear_b, float* out_scores);

/* Stage-1 alone, for parity tests against MLM_PLL/preprocess.py:9-30:
 * expands the hypotheses into the packed masked copies.
 * out_ids      DEVICE int32[sum L*(L+2)]  input_ids of every copy, packed
 * out_mask_pos DEVICE int32[sum L]        mask_pos of every copy (1-based incl. [CLS])
 * out_labels   DEVICE int32[sum L]        labels[mask_pos] of every copy        */
int pllb_expand(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
                int32_t n_hyp, int32_t* out_ids, int32_t* out_mask_pos, int32_t* out_labels,
                void* stream);

int pllb_get_stats(pllb_handle h, pllb_stats* out);
int pllb_reset_stats(pllb_handle h);
/* enable=1: bracket GEMM launches with CUDA events on the launch stream so
 * last_gemm_ms is filled (adds event-record overhead only). */
int pllb_set_timing(pllb_handle h, int enable);
/* Device time (ms) per GEMM kind of the last timed pllb_score call and FLOPs issued per
 * kind since the last reset.  Order: QKV, attention-output, FFN1, FFN2, head transform,
 * decoder(+logsumexp).  Either pointer may be NULL. */
int pllb_get_gemm_breakdown(pllb_handle h, float* ms6, double* flops6);

/* ---- Debug / parity hooks (encoder internals; used by tests only) ---------
 * C[M,N] = A[M,K] * W[N,K]^T + bias[N], through the tcgen05 GEMM kernel.
 * A, W: DEVICE bf16 (raw uint16) row-major; bias fp32; epilogue:
 *   0 = bias -> bf16 out, 1 = bias+GELU(erf) -> bf16 out,
 *   2 = bias -> fp32 out, 3 = bias+GELU(erf) -> fp32 out.
 * N % 256 == 0, K % 64 == 0. */
int pllb_debug_gemm(const uint16_t* A, const uint16_t* W, const float* bias, void* C,
                    int32_t M, int32_t N, int32_t K, int32_t epilogue, void* stream);
/* Same with an explicit operand type: 0 = A and W bf16, 1 = A and W IEEE fp16 (raw uint16);
 * 16-bit outputs are written in the operand type. */
int pllb_debug_gemm_dt(const uint16_t* A, const uint16_t* W, const float* bias, void* C,
                       int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t operand_dtype, void* stream);
/* Same arithmetic through the plain SIMT validation kernel (slow). */
int pllb_debug_gemm_simt(const uint16_t* A, const uint16_t* W, const float* bias, void* C,
                         int32_t M, int32_t N, int32_t K, int32_t epilogue, void* stream);
/* Final hidden states (fp32 [tokens, hidden]) of the packed masked copies of
 * the given hypotheses after `upto_layer` encoder layers (0 = embeddings). */
int pllb_debug_hidden(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets,
                      int32_t n_hyp, int32_t upto_layer, float* out_hidden, void* stream);

/* Kernel hooks of the training path (the non-GEMM kernels the MLM, RescoreBert and CorrectBart
 * trainers share; used by tests only).  Every pointer is a caller DEVICE buffer; the launches are
 * those of a training step.  bf16 buffers are raw uint16.  Dropout: probability p in [0, 1) over the
 * DEVICE uint64 *seed (may be NULL when p == 0) at dropout site `site`, as in a step.  Bad scalars or
 * pointers, H outside {256, 512, 768, 1024}, T outside [1, 512], and device index arrays out of range
 * (n_valid outside [1, T], ids outside [0, vocab), labels outside [0, V) and not -100 where allowed)
 * return PLLB_ERR_INVALID before anything is launched; the index checks synchronise the stream.  The
 * attention hooks also refuse misaligned pointers: bf16 q / k / v (qkv) and fp32 dctx on 16 bytes,
 * fp32 dq / dk / dv (dqkv) on 8, the rest on 4.
 *
 * Padded self-attention of B sequences of T rows, NH = H / 64 heads: qkv bf16 [B*T, 3H] (q | k | v),
 * n_valid int32[B].  Forward: ctx bf16 [B*T, H], lse fp32 [B*T*NH].  With dctx (fp32 [B*T, H]) also the
 * backward: dqkv fp32 [B*T, 3H], Dscratch fp32 [B*T*NH] (D = sum_j P dP of every (row, head)). */
int pllb_debug_train_attn(const uint16_t* qkv, const int32_t* n_valid, int32_t B, int32_t T, int32_t H,
                          const float* dctx, const uint64_t* seed, float p, uint32_t site, uint16_t* ctx,
                          float* lse, float* dqkv, float* Dscratch, void* stream);
/* The decoder's attention: Tq query rows (q, row stride ldq) over Tk key / value rows (k, v, row stride
 * ldkv) per sequence.  causal != 0: Tq == Tk, query i sees keys <= i (n_valid unused); otherwise keys
 * < n_valid[b].  ctx bf16 [B*Tq, NH*64], lse [B*Tq*NH]; with dctx (fp32 [B*Tq, NH*64]) also dq (row
 * stride lddq), dk and dv (row stride lddkv) and Dscratch [B*Tq*NH].  ldq % 8 == ldkv % 8 == 0. */
int pllb_debug_s2s_attn(const uint16_t* q, const uint16_t* k, const uint16_t* v, int32_t ldq, int32_t ldkv,
                        const int32_t* n_valid, int32_t B, int32_t Tq, int32_t Tk, int32_t NH, int32_t causal,
                        const float* dctx, const uint64_t* seed, float p, uint32_t site, uint16_t* ctx, float* lse,
                        float* dq, int32_t lddq, float* dk, float* dv, int32_t lddkv, float* Dscratch, void* stream);
/* LayerNorm forward over R rows of H, saving xhat and rstd (either may be NULL in form 0).
 * form 0: LN(dropout(y) + res)            (res may be NULL; out32 / out16 may be NULL)
 * form 1: dropout(LN(word[ids[r]] + pos[r % T] + type[0]))        (BERT embeddings)
 * form 2: dropout(LN(word[ids[r]] * embed_scale + pos[r % T]))    (BART embeddings; every output required) */
int pllb_debug_train_ln_fwd(int32_t form, const float* y, const float* res, const int32_t* ids, int32_t T,
                            const float* word, int32_t vocab, const float* pos, const float* type, float embed_scale,
                            const float* g, const float* b, float eps, int32_t R, int32_t H, const uint64_t* seed,
                            float p, uint32_t site, float* out32, uint16_t* out16, float* xhat, float* rstd,
                            void* stream);
/* LayerNorm backward: dy <- (dy + add) [* mask site_in]; dz = the input gradient; dz_drop = dz [* mask
 * site_out] (may be NULL).  add may be NULL or alias dz; site -1 = no mask. */
int pllb_debug_train_ln_bwd(float* dy, const float* add, const float* g, const float* xhat, const float* rstd,
                            int32_t R, int32_t H, const uint64_t* seed, float p, int32_t site_in, int32_t site_out,
                            float* dz, float* dz_drop, void* stream);
/* Cross entropy over the first V of Vp logit columns (fp32 [R, Vp]): loss_rows [R]; dlogits bf16 [R, Vp]
 * = softmax - onehot, 0 past V (may be NULL).  ignore_index 0: out_loss[0] = the mean loss.
 * ignore_index != 0: label -100 gives loss 0 and a zero dlogits row; out_loss[0] = the mean over the N
 * labelled rows, out_loss[1] = 1 / N. */
int pllb_debug_train_ce(const float* logits, const int32_t* labels, int32_t R, int32_t V, int32_t Vp,
                        int32_t ignore_index, float* loss_rows, uint16_t* dlogits, float* out_loss, void* stream);
/* Embedding backward from dz fp32 [B*T, H]: dpos [pos_rows, H] (rows >= T zero); dword [vocab, H] += the
 * rows of each id except pad_id.  form 0 (BERT): dtype0 [H] = the column sums (scratch: 128 * H floats
 * or NULL).  form 1 (BART): dz is scaled by `scale` in place before the word scatter. */
int pllb_debug_train_embed_bwd(int32_t form, float* dz, const int32_t* ids, int32_t B, int32_t T, int32_t H,
                               int32_t pos_rows, int32_t pad_id, float scale, float* dword, int32_t vocab,
                               float* dpos, float* dtype0, float* scratch, void* stream);
/* Column sums of dy [R, C] (fp32, or bf16 when dy_bf16): out_sum[c] = sum_r dy, out_dot[c] = sum_r
 * dy * xhat (either may be NULL).  scratch: 128 * C floats for the row-sliced form, or NULL. */
int pllb_debug_train_colsum(const void* dy, int32_t dy_bf16, const float* xhat, int32_t R, int32_t C,
                            float* out_sum, float* out_dot, float* scratch, void* stream);
/* src [R, C] (fp32, or bf16 when src_bf16) -> dst16 bf16 [R, C] and / or dstT bf16 [C, Rp], columns
 * >= R of dstT zero.  Rp >= R. */
int pllb_debug_train_cast_transpose(const void* src, int32_t src_bf16, int32_t R, int32_t C, int32_t Rp,
                                    uint16_t* dst16, uint16_t* dstT, void* stream);
/* GELU (erf form) of f [n]: out16 bf16 and / or out32; then dg[i] *= GELU'(f[i]) when dg != NULL. */
int pllb_debug_train_gelu(const float* f, int64_t n, uint16_t* out16, float* out32, float* dg, void* stream);

/* ---- BERTScore minimum-Bayes-risk (RMBR): replaces bert_score.score(cands, refs, lang="zh") inside
 * RMBR/utility_functions.py:9-23 (BertScoreFunction).  RMBR/ and bert_score are not in the reference
 * tree, so this is the library's own contract, following bert_score with its default arguments
 * (idf=False, no baseline rescaling, bert-base-chinese truncated to num_layers encoder layers; its
 * model table gives 8):
 *   E(t)    fp32 output of encoder layer num_layers for all L+2 positions of [CLS] t [SEP]
 *           (bert_score's model(...)[0] after model.encoder.layer = layer[:num_layers]).
 *   R(c, r) = mean over x in r[1 .. T_r-2] of max over y in c[0 .. T_c-1] of cos(E_r[x], E_c[y])
 *           The reference's [CLS] / [SEP] carry weight 0; the candidate's take part in the max
 *           (bert_score's greedy_cos_idf with uniform idf).  R = 0 when either sentence is empty
 *           (T == 2).  The max runs over real positions only: bert_score multiplies the similarity
 *           matrix by the padding mask, so where every real cosine of a column is negative its padded
 *           batch returns 0 instead (DESIGN.md §3.9).
 *   P(c, r) = R(r, c): precision is the same call with the roles swapped.
 *
 * Embedding pass: hyp_tokens / hyp_offsets as in pllb_score.  num_layers in [0, desc.num_layers]
 * (0 = the embedding LayerNorm output).  out_hidden DEVICE float[sum (L+2), hidden] row-major;
 * sequence i starts at row (hyp_offsets[i] - hyp_offsets[0]) + 2 i.  A sequence longer than
 * max_position returns PLLB_ERR_TOO_LONG.  The handle may be created without MLM head weights.
 * Asynchronous on `stream` under the one-stream rule of pllb_score. */
int pllb_embed(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets, int32_t n_hyp,
               int32_t num_layers, float* out_hidden, void* stream);
/* Pair recall: out_recall[p] = R(sequence cand[p], sequence ref[p]) for sequences whose rows lie in
 * emb (DEVICE fp32 [rows, hidden], 16-byte aligned): sequence i is rows row_off[i] .. row_off[i+1]-1.
 * row_off HOST int64[n_seq+1], cand / ref HOST int32[n_pairs] (control metadata, validated here:
 * an index outside [0, n_seq), non-monotone offsets or a sequence with fewer than 2 rows return
 * PLLB_ERR_INVALID) are copied through the handle's pinned metadata buffer.  Consecutive pairs with
 * the same candidate share one CTA, which keeps the candidate's rows on chip: emit pairs grouped by
 * candidate (mbr_decode does).  fp32 throughout, one launch, bit-deterministic.  Asynchronous on
 * `stream` under the one-stream rule of pllb_score. */
int pllb_bertscore(pllb_handle h, const float* emb, const int64_t* row_off, int32_t n_seq, const int32_t* cand,
                   const int32_t* ref, int32_t n_pairs, float* out_recall, void* stream);

/* ---- Text front end: replaces BertTokenizer.tokenize + convert_tokens_to_ids
 * (MLM_PLL/preprocess.py:10,16-27,34) for hypotheses made of CJK ideographs,
 * punctuation and whitespace, where BERT's BasicTokenizer makes every character
 * its own token.  Strings are packed Unicode code points (HOST arrays).
 * table int32[table_size], indexed by code point:
 *   >= 0              wordpiece id of the character as a token ([UNK] if not in the vocab)
 *   PLLB_TOK_SPACE    whitespace: separates, emits nothing
 *   PLLB_TOK_REMOVED  control character, U+0000, U+FFFD: removed
 *   PLLB_TOK_WORD     part of a word run (Latin, digits, kana, marks ...): the hypothesis
 *                     needs the host wordpiece tokenizer; needs_host[h] = 1 and it gets
 *                     0 tokens here.  Code points >= table_size count as PLLB_TOK_WORD.
 * out_ids: capacity cp_off[n_hyp]; out_off int64[n_hyp+1]; needs_host uint8[n_hyp]. */
#define PLLB_TOK_SPACE (-1)
#define PLLB_TOK_REMOVED (-2)
#define PLLB_TOK_WORD (-3)
int pllb_tokenize_host(const int32_t* table, int32_t table_size, const int32_t* cp,
                       const int64_t* cp_off, int32_t n_hyp, int32_t* out_ids,
                       int64_t* out_off, uint8_t* needs_host);

/* ---- Levenshtein: replaces jiwer.cer's per-pair edit distance at
 * rescore.py:40,118 (and espnet_data/preprocess/main.py:59-60).
 * Strings are packed arrays of Unicode code points.
 * pair i compares ref[pair_ref[i]] with hyp i.  out_dist[i] = edit distance. */
int pllb_levenshtein(const int32_t* ref_cp, const int64_t* ref_off,
                     const int32_t* hyp_cp, const int64_t* hyp_off,
                     const int32_t* pair_ref, int32_t n_pairs, int32_t max_len,
                     int32_t* out_dist, void* stream);
int pllb_levenshtein_host(const int32_t* ref_cp, const int64_t* ref_off, int32_t n_ref,
                          const int32_t* hyp_cp, const int64_t* hyp_off,
                          const int32_t* pair_ref, int32_t n_pairs, int32_t* out_dist);

/* ---- Edit-operation alignment: the Levenshtein DP with backtrace of the reference's
 * espnet_data/preprocess/align.py (hyp_alignment.json) and the U/S/I/D counts of its
 * statistic/error_type_count.py.  DESIGN.md §3.10.
 * Symbols are opaque int32 (the Python side passes code points of the stripped strings, as
 * for pllb_levenshtein, so S + I + D is that call's distance; token ids work too).  Same
 * packing as pllb_levenshtein: pair i aligns ref[pair_ref[i]] (i indexes it) with hyp i (j).
 * D[i][j] is the unit-cost table of pllb_levenshtein.  The backtrace starts at (na, nb) and
 * at each cell takes the first predecessor in this order that attains D[i][j]:
 *   1. diagonal: 'U' if the symbols are equal, 'S' otherwise;
 *   2. up (i-1): 'I', a reference symbol with no hypothesis counterpart;
 *   3. left (j-1): 'D', a hypothesis symbol with no reference counterpart.
 * The letters are the reference's and the reverse of jiwer's naming ('I' is what jiwer calls a
 * deletion, 'D' an insertion).  Pinned by the reference's own docstring examples
 * (tests/golden/levenshtein_meta.json): the letters, and diagonal before left on a tie.  Up
 * before left is this project's reading of align.py; no known-answer test pins it.
 * ops_off int64[n_pairs+1]: pair i owns out_ops[ops_off[i] .. ops_off[i+1]), at least na + nb
 * bytes.  The kernel writes the ops as ASCII 'U' 'S' 'I' 'D' in forward order (first symbol
 * first) at the start of the slot and zeroes the slot's remaining bytes up to na + nb;
 * out_n_ops[i] = number of ops, in [max(na, nb), na + nb]; out_counts int32[n_pairs*4] =
 * (U, S, I, D) of pair i.  A side longer than 1024 symbols returns PLLB_ERR_TOO_LONG.
 * Integer only, no atomics, bit-deterministic.
 * pllb_align: DEVICE arrays, asynchronous on `stream`.  max_len >= every na and nb (a pair
 * above it gets out_n_ops = -1 and zero counts).  When max_len > 64 the codes go to the calling
 * thread's device scratch region, which the *_host entry points share: issue those calls from
 * one thread on one stream, or synchronise between them.
 * pllb_align_host: HOST arrays; validates pair_ref, the offsets (non-negative, ascending, slots
 * of at least na + nb) with PLLB_ERR_INVALID and the lengths with PLLB_ERR_TOO_LONG, copies
 * through the scratch region and returns when the results are in host memory.  Bytes of a slot
 * past na + nb are zeroed too. */
int pllb_align(const int32_t* ref_cp, const int64_t* ref_off,
               const int32_t* hyp_cp, const int64_t* hyp_off,
               const int32_t* pair_ref, int32_t n_pairs, int32_t max_len,
               const int64_t* ops_off, uint8_t* out_ops, int32_t* out_n_ops,
               int32_t* out_counts, void* stream);
int pllb_align_host(const int32_t* ref_cp, const int64_t* ref_off, int32_t n_ref,
                    const int32_t* hyp_cp, const int64_t* hyp_off,
                    const int32_t* pair_ref, int32_t n_pairs, const int64_t* ops_off,
                    uint8_t* out_ops, int32_t* out_n_ops, int32_t* out_counts);

/* ---- Combiner: replaces rescore.py:47-58 (rescore + get_highest_score_hyp)
 * and the per-weight CER numerator of rescore.py:37-43 (find_best_weight).
 * variant 0: (1-w)*am/len + w*lm/len   (rescore.py:51, current source)
 * variant 1: (1-w)*am     + w*lm       (rescore_result/MLM_PLL/rescore.log:28)
 * variant 2: (1-w)*am/len + w*lm       (rescore_result/RMBR/BertScore/rescore_mbr_normalize.log:29)
 * All arrays [N, n_best] row-major; fp64, no FMA contraction, numpy op order.
 * out_argmax int32[W, N]; out_edit_sum int64[W] = sum_u dist[u, argmax]. */
int pllb_rescore_sweep(const double* am, const double* lm, const int64_t* len,
                       const int32_t* dist, int32_t N, int32_t n_best,
                       const double* weights, int32_t W, int32_t variant,
                       int32_t* out_argmax, int64_t* out_edit_sum, void* stream);
int pllb_rescore_sweep_host(const double* am, const double* lm, const int64_t* len,
                            const int32_t* dist, int32_t N, int32_t n_best,
                            const double* weights, int32_t W, int32_t variant,
                            int32_t* out_argmax, int64_t* out_edit_sum);
/* The [N, n_best] score matrix for one weight (rescore.py:47-53), DEVICE fp64. */
int pllb_rescore_scores(const double* am, const double* lm, const int64_t* len,
                        int32_t N, int32_t n_best, double weight, int32_t variant,
                        double* out_scores, void* stream);

/* ---- MLM fine-tuning: replaces the train_mode=True branch of run_one_epoch
 * (MLM_PLL/main.py:73-99: BertForMaskedLM.forward with labels, loss.backward(),
 * torch.optim.AdamW.step(), zero_grad) and its loss-only twin (train_mode=False,
 * do_scoring=False — the dev pass of mlm_finetune_bert, MLM_PLL/main.py:146-153).
 * A batch is what collate (MLM_PLL/main.py:28-54) builds: B sequences zero-padded to T
 * positions; the loss is CrossEntropyLoss() over ALL B*T positions (labels are the whole
 * unmasked sequence, pad positions carry label 0 = [PAD]; nothing is ignored).
 * fp32 master weights / gradients / Adam moments; bf16 operands, fp32 accumulation in
 * every GEMM (forward, dgrad, wgrad).  The decoder weight is tied to the word embeddings
 * and the decoder bias is cls.predictions.bias. */
typedef struct pllb_train_desc {
  float lr;                 /* config.lr (MLM_PLL/config/train.yaml:5: 1e-5)          */
  float beta1, beta2;       /* torch.optim.AdamW defaults 0.9, 0.999                  */
  float adam_eps;           /* 1e-8                                                    */
  float weight_decay;       /* 0.01, applied to EVERY parameter (model.parameters())  */
  float hidden_dropout;     /* BertConfig.hidden_dropout_prob (0.1); 0 for parity runs */
  float attention_dropout;  /* BertConfig.attention_probs_dropout_prob (0.1)          */
  uint64_t seed;            /* dropout stream (the masks are a stateless hash)        */
  int32_t pad_id;           /* BertConfig.pad_token_id (0): the embedding lookup sends
                               no gradient to this row (nn.Embedding padding_idx)     */
  int32_t max_rows;         /* capacity: B * T of the largest batch                    */
  int32_t max_seq;          /* capacity: largest T (<= max_position, <= 512)           */
} pllb_train_desc;

typedef struct pllb_trainer_ctx* pllb_trainer;

/* weights: DEVICE fp32 state_dict tensors (copied; the MLM head is required). */
int pllb_train_create(pllb_trainer* out, const pllb_model_desc* desc, const pllb_weights* weights,
                      const pllb_train_desc* train, int device);
int pllb_train_destroy(pllb_trainer t);
int64_t pllb_train_workspace_bytes(pllb_trainer t);
int64_t pllb_train_kernel_launches(pllb_trainer t);
/* Steps that ran as a replay of a captured CUDA graph (a batch shape (B, T, mode) runs eagerly
 * once, is captured on its second occurrence and replayed afterwards; PLLB_TRAIN_GRAPH=0 disables). */
int64_t pllb_train_graph_replays(pllb_trainer t);
/* A fresh optimizer: zero moments, step count 0, learning rate lr — the reference
 * re-creates AdamW at the start of every epoch (MLM_PLL/main.py:76). */
int pllb_train_reset_optimizer(pllb_trainer t, float lr);
/* One batch, HOST buffers.  input_ids, labels: int32[B*T] row-major (zero-padded as collate
 * does); n_valid: int32[B], the number of leading positions with attention_mask 1.
 * mode 0: loss only (model.eval(): no dropout, no update);
 * mode 1: forward (dropout active) + backward + AdamW step;
 * mode 2: forward + backward, no update (gradients stay readable: parity tests).
 * out_loss: the batch loss (output.loss.item(), MLM_PLL/main.py:109).  Synchronises. */
int pllb_train_step_host(pllb_trainer t, const int32_t* input_ids, const int32_t* n_valid,
                         const int32_t* labels, int32_t B, int32_t T, int32_t mode, float* out_loss);
/* Per-position losses of the last step, HOST float[B*T]: loss[b*T + t] = -log_softmax(logits[b, t])[labels[b, t]].
 * With the for_scoring rows of preprocess.py (labels = the unmasked sequence) the entry at the row's mask_pos is
 * minus the PLL term the scoring branch adds (MLM_PLL/main.py:101-107) — this is what makes
 * run_one_epoch(train_mode=..., do_scoring=True) work on a trainer. */
int pllb_train_row_losses_host(pllb_trainer t, float* out, int32_t n);
/* Writes the fp32 master weights (model.state_dict(), MLM_PLL/main.py:155) / the gradients of
 * the last mode-1/2 step into the caller's DEVICE tensors; a NULL pointer skips that tensor;
 * q/k/v are un-stacked; decoder_w is written only if it is not the word_emb pointer. */
int pllb_train_export(pllb_trainer t, const pllb_weights* dst);
int pllb_train_export_grads(pllb_trainer t, const pllb_weights* dst);

/* ---- RescoreBert distillation: the student of RescoreBert/main.py (BertModel, then Linear(H, 1)
 * on the [CLS] state; the scorer is pllb_score_cls) trained on the teacher's PLLs.  The
 * reference's training script is not part of the reference tree, so the losses below are this
 * library's contract, pinned by an autograd restatement (oracle/rescorebert_train_oracle.py), not
 * by a reference golden.  A batch is B hypotheses of whole utterances, zero-padded to T positions;
 * the hypotheses of one utterance are contiguous rows and form one group (G groups).
 *   s_i  = linear_w . h_L[i, 0, :] + linear_b      (fp32 last-layer output at [CLS])
 *   MD   = (1/B) sum_i (s_i - y_i)^2               (nn.MSELoss(); y = teacher PLL)
 *   P    = softmax over the group of (am_weight * a + s)   (a = AM score)
 *   MWER = (1/G) sum_g sum_{i in g} P_i (e_i - mean_g e)   (e = per-hypothesis CER)
 *   loss = md_weight * MD + mwer_weight * MWER
 * A group of one hypothesis has P = 1 and contributes 0 to MWER and to its gradient; it still
 * counts in G.  Encoder, optimizer, dropout and graphs are those of the MLM trainer above; AdamW
 * (weight decay on every parameter) also updates linear_w and linear_b.  The pooler of BertModel
 * gets no gradient and is not held here. */
typedef struct pllb_cls_loss_desc {
  float md_weight;          /* >= 0 */
  float mwer_weight;        /* >= 0; 0 = MD alone */
  float am_weight;          /* scale of the AM score inside the MWER softmax */
} pllb_cls_loss_desc;

/* weights: DEVICE fp32 encoder tensors (the head pointers are ignored); linear_w DEVICE fp32 [H],
 * linear_b DEVICE fp32 [1] (copied).  The handle works with pllb_train_destroy, _reset_optimizer,
 * _workspace_bytes, _kernel_launches and _graph_replays; pllb_train_step_host, _row_losses_host and
 * _export* reject it (PLLB_ERR_INVALID), as the pllb_cls_train_* calls reject an MLM trainer. */
int pllb_cls_train_create(pllb_trainer* out, const pllb_model_desc* desc, const pllb_weights* weights,
                          const float* linear_w, const float* linear_b, const pllb_train_desc* train,
                          const pllb_cls_loss_desc* loss, int device);
/* One batch, HOST buffers.  input_ids int32[B*T] ([CLS] t [SEP], zero-padded); n_valid int32[B];
 * group int32[B]: 0 for the first row, then each entry equal to the previous one or one more;
 * target / am / err float[B], finite.  mode as in pllb_train_step_host.  out_loss: the batch loss;
 * out_scores: float[B] per-hypothesis scores of this forward pass (may be NULL).  Synchronises. */
int pllb_cls_train_step_host(pllb_trainer t, const int32_t* input_ids, const int32_t* n_valid,
                             const int32_t* group, const float* target, const float* am,
                             const float* err, int32_t B, int32_t T, int32_t mode, float* out_loss,
                             float* out_scores);
/* Encoder tensors into the caller's DEVICE tensors as pllb_train_export* (NULL skips a tensor),
 * linear_w [H] and linear_b [1] DEVICE. */
int pllb_cls_train_export(pllb_trainer t, const pllb_weights* dst, float* linear_w, float* linear_b);
int pllb_cls_train_export_grads(pllb_trainer t, const pllb_weights* dst, float* linear_w, float* linear_b);

/* ---- Greedy seq2seq generation: CorrectBart's one_hyp correction (CorrectBart/ in the reference: a
 * BartForConditionalGeneration reads the 1-best hypothesis and generate()s a corrected sentence).
 * DESIGN.md §3.11.  The model is BART with post-LN layers (bart-base): no final encoder / decoder
 * layer_norm, activation "gelu", head dim 64, hidden and both FFN widths multiples of 256, every
 * LayerNorm with the same eps (1e-5).
 *   encoder: [CLS] t [SEP] (cls_id / sep_id), token rows * embed_scale + positions (row i + 2 of
 *            embed_positions), layernorm_embedding, the BERT-form post-LN layers.  It runs through
 *            the pllb_create / pllb_embed path with a zero token-type row.
 *   decoder: position 0 holds decoder_start_id.  The step that writes position t feeds the token at
 *            t - 1 (token row * embed_scale + embed_positions row t - 1 + 2, layernorm_embedding), runs
 *            every layer against the KV cache of positions 0 .. t - 1 and the sentence's encoder rows,
 *            and takes logits = h . shared^T + final_logits_bias (embed_scale does not touch the head).
 *   choice:  the first index of the maximum (torch.argmax); forced_bos_id replaces it at t = 1,
 *            forced_eos_id at t = max_length - 1 (the EOS one wins when both apply); a sentence that
 *            has emitted eos_id emits pad_id from then on.  Decoding stops when every sentence has
 *            emitted EOS or position max_length - 1 has been written.  This equals
 *            generate(num_beams=1, do_sample=False, max_length=...) with these settings.
 * Operand type (operand_dtype): 0 = bf16, 1 = IEEE fp16 for every GEMM operand, the self-attention KV
 * cache and the cross-attention K/V; fp32 accumulation, fp32 residual stream, fp32 softmax. */
typedef struct pllb_s2s_desc {
  int32_t enc_layers, dec_layers;
  int32_t hidden;              /* d_model: 256 / 512 / 768 / 1024                                  */
  int32_t num_heads;           /* hidden / 64, both stacks                                         */
  int32_t enc_intermediate;    /* encoder_ffn_dim, multiple of 256                                 */
  int32_t dec_intermediate;    /* decoder_ffn_dim, multiple of 256                                 */
  int32_t vocab;
  int32_t enc_max_position;    /* max_position_embeddings: rows of encoder embed_positions - 2     */
  int32_t dec_max_position;    /* same for the decoder                                             */
  float   ln_eps;              /* 1e-5                                                             */
  float   embed_scale;         /* sqrt(d_model) with scale_embedding, else 1                       */
  int32_t cls_id, sep_id;      /* the encoder input's [CLS] / [SEP] ids                            */
  int32_t operand_dtype;       /* 0 bf16, 1 fp16                                                   */
} pllb_s2s_desc;

/* One decoder layer; DEVICE fp32 tensors in nn.Linear layout (model.decoder.layers.{i}.*). */
typedef struct pllb_dec_layer_weights {
  const float *q_w, *q_b, *k_w, *k_b, *v_w, *v_b, *o_w, *o_b;         /* self_attn.{q,k,v,out}_proj        */
  const float *self_ln_g, *self_ln_b;                                  /* self_attn_layer_norm              */
  const float *cq_w, *cq_b, *ck_w, *ck_b, *cv_w, *cv_b, *co_w, *co_b; /* encoder_attn.{q,k,v,out}_proj     */
  const float *cross_ln_g, *cross_ln_b;                                /* encoder_attn_layer_norm           */
  const float *ff1_w, *ff1_b, *ff2_w, *ff2_b;                          /* fc1, fc2                          */
  const float *final_ln_g, *final_ln_b;                                /* final_layer_norm                  */
} pllb_dec_layer_weights;

typedef struct pllb_s2s_weights {
  /* encoder, DEVICE fp32: word_emb and type_emb are ignored (the token table is `shared`, the
   * token-type row is zero); pos_emb = model.encoder.embed_positions.weight + 2 * hidden (the offset
   * rows skipped); emb_ln_* = model.encoder.layernorm_embedding; layers = model.encoder.layers
   * (self_attn.{q,k,v,out}_proj, self_attn_layer_norm, fc1, fc2, final_layer_norm); head pointers
   * ignored. */
  pllb_weights enc;
  const pllb_dec_layer_weights* dec_layers;   /* HOST array of dec_layers structs                 */
  const float* shared;                        /* model.shared.weight [vocab, hidden], unscaled     */
  const float* dec_pos_emb;                   /* model.decoder.embed_positions.weight + 2 * hidden */
  const float *dec_emb_ln_g, *dec_emb_ln_b;   /* model.decoder.layernorm_embedding                 */
  const float* final_logits_bias;             /* [vocab]                                           */
} pllb_s2s_weights;

/* generate() settings.  Everything generate() would apply beyond greedy decoding is rejected with
 * PLLB_ERR_INVALID: num_beams != 1 (beam search is pllb_generate_beam), do_sample != 0,
 * no_repeat_ngram_size != 0, min_length != 0, repetition_penalty != 1. */
typedef struct pllb_gen_desc {
  int32_t max_length;          /* 2 <= max_length <= dec_max_position                              */
  int32_t decoder_start_id, eos_id, pad_id;
  int32_t forced_bos_id;       /* -1 = none */
  int32_t forced_eos_id;       /* -1 = none */
  int32_t num_beams, do_sample, no_repeat_ngram_size, min_length;
  float   repetition_penalty;
} pllb_gen_desc;

/* Counters since create (or the last reset) and, with timing enabled, the device time of the last
 * pllb_generate call split by phase. */
typedef struct pllb_s2s_stats {
  int64_t kernel_launches;     /* kernels of this library launched                                 */
  int64_t steps;               /* decoder steps run (summed over chunks)                           */
  int64_t chunks;
  int64_t sentences;
  double  gemm_flops;          /* algorithmic GEMM FLOPs (encoder, cross K/V, decoder, head)       */
  float   enc_ms, cross_kv_ms, dec_layers_ms, head_ms;   /* last call, timing enabled               */
  float   total_ms;                                      /* last call, timing enabled               */
} pllb_s2s_stats;

typedef struct pllb_s2s_ctx* pllb_s2s;

/* weights are copied (16-bit operands, fp32 rest).  max_rows bounds the sentences decoded together
 * per internal chunk (0 = 8192); the per-call workspace grows with max_rows * max_length: the KV
 * cache alone is rows * max_length * 2 * hidden * dec_layers * 2 bytes.  Results do not depend on
 * max_rows. */
int pllb_s2s_create(pllb_s2s* out, const pllb_s2s_desc* desc, const pllb_s2s_weights* weights, int32_t max_rows,
                    int device);
int pllb_s2s_destroy(pllb_s2s h);
int64_t pllb_s2s_workspace_bytes(pllb_s2s h);
int pllb_s2s_set_timing(pllb_s2s h, int enable);
int pllb_s2s_get_stats(pllb_s2s h, pllb_s2s_stats* out);
int pllb_s2s_reset_stats(pllb_s2s h);

/* tokens DEVICE int32 (ids in [0, vocab): pllb_generate_host checks them), no specials; sentence i is
 * tokens[offsets[i] .. offsets[i+1]); offsets HOST int64[n+1].  A sentence with more than
 * enc_max_position - 2 tokens returns PLLB_ERR_TOO_LONG.
 * out_ids   DEVICE int32[n * max_length]: sentence i's ids at [i * max_length, ...), position 0 = start
 *           token, pad_id after the end (generate() returns the same up to its own padding width);
 * out_len   DEVICE int32[n]: positions up to and including EOS (max_length when none was emitted);
 * out_logit DEVICE float[n * max_length] or NULL: fp32 logit of each chosen token (at a forced position
 *           the logit of the forced token), 0 at position 0 and at pad positions.
 * Runs on `stream` and waits for it once per decoder step (the count of finished sentences decides
 * whether to continue): the call returns when the results are complete. */
int pllb_generate(pllb_s2s h, const pllb_gen_desc* gen, const int32_t* tokens, const int64_t* offsets, int32_t n,
                  int32_t* out_ids, int32_t* out_len, float* out_logit, void* stream);
int pllb_generate_host(pllb_s2s h, const pllb_gen_desc* gen, const int32_t* tokens, const int64_t* offsets, int32_t n,
                       int32_t* out_ids, int32_t* out_len, float* out_logit);

/* ---- Beam search (DESIGN.md §3.12): generate(num_beams=K, do_sample=False) of transformers 5.5.0
 * (GenerationMixin._beam_search) with one EOS id.  K = pllb_gen_desc.num_beams, 2 <= K <= 8,
 * vocab >= 2K, K * max_length <= 12288; every other pllb_gen_desc field is checked as pllb_generate
 * checks it.  t is the position being written (the start token is at 0), ML = max_length.
 *  1. logp = log_softmax(fp32 logits) of each running beam, logits as greedy; forced BOS (t = 1) and
 *     forced EOS (t = ML - 1, wins when both apply) set the forced id to 0 and every other id to -inf.
 *  2. cand = logp + running_score[beam] (fp32); running scores start [0, -1e9, ...].  The step keeps
 *     the top 2K of the K * V candidates of a sentence.
 *  3. A candidate hits the stopping criteria when its token is eos_id or t = ML - 1.
 *  4. The next running beams are the top K of cand + hit * -1e9 (fp32), each with its parent beam.
 *  5. K finished slots per sentence start at score -1e9, not finished.  Candidate c of the 2K enters
 *     with cand / (float)(t ** length_penalty), then -1e9 is added (fp32, in this order) when every
 *     slot is finished and early_stopping is 1; when the early-stop heuristic is satisfied; and
 *     unless c < K and c hit.  The new slots are the top K of [old slots ++ 2K candidates].
 *  6. Early-stop heuristic, after the step: it stays unsatisfied only while it was unsatisfied and,
 *     for some slot, best_running / L ** length_penalty > (slot finished ? min(slot scores) : -1e9),
 *     with L = t (L = ML - 1 when early_stopping is 2 and length_penalty > 0).
 *  7. A sentence is frozen once the heuristic is satisfied, or early_stopping is 1 and every slot is
 *     finished; its slots cannot change from then on.  Decoding stops when every sentence is frozen
 *     or position ML - 1 has been written.
 *  8. The result is the best num_return_sequences slots in descending score order.
 *  9. Ties: higher value first, then lower flat index (beam * V + token; slot before candidate).
 * max_rows of pllb_s2s_create counts decoder rows (beams): a chunk holds max_rows / K sentences, and
 * max_rows < K is PLLB_ERR_INVALID.  Results do not depend on max_rows.  The time of the selection
 * kernel is part of pllb_s2s_stats.head_ms. */
typedef struct pllb_beam_desc {
  int32_t num_return_sequences;   /* 1 <= r <= num_beams                                             */
  float   length_penalty;         /* finite                                                          */
  int32_t early_stopping;         /* 0 False, 1 True, 2 "never"                                      */
} pllb_beam_desc;

/* tokens / offsets as pllb_generate.  Outputs (DEVICE):
 * out_ids   int32[n * r * max_length]: hypothesis k of sentence i at [(i * r + k) * max_length, ...),
 *           position 0 = start token, pad_id after the end;
 * out_len   int32[n * r]: positions up to and including EOS, start included;
 * out_score float[n * r]: the finished-slot score (sum of logp / (len - 1) ** length_penalty). */
int pllb_generate_beam(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, const int32_t* tokens,
                       const int64_t* offsets, int32_t n, int32_t* out_ids, int32_t* out_len, float* out_score,
                       void* stream);
/* The same with HOST tokens and outputs; token ids are checked against the vocabulary. */
int pllb_generate_beam_host(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, const int32_t* tokens,
                            const int64_t* offsets, int32_t n, int32_t* out_ids, int32_t* out_len, float* out_score);
/* Test hook: the selection alone on given decoder outputs.  hidden HOST fp32 [steps = max_length - 1,
 * n * K, hidden] (row i * K + b is beam b of sentence i at that step), rounded to the operand type and
 * fed to the LM head with EPI_TOPK, beam_select_kernel and the bookkeeping; no decoder layers, and
 * n * K <= max_rows.  HOST outputs as pllb_generate_beam_host, plus out_parent int32[steps, n * K]
 * (chunk row of each running beam's parent) and out_run_score float[steps, n * K]; steps not run
 * hold -1 / 0. */
int pllb_s2s_debug_beam_replay(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, int32_t n,
                               const float* hidden, int32_t steps, int32_t* out_ids, int32_t* out_len,
                               float* out_score, int32_t* out_parent, float* out_run_score);

/* ---- CorrectBart fine-tuning (DESIGN.md §3.13): one step is what transformers 5.5.0 computes for
 * BartForConditionalGeneration.forward(input_ids, attention_mask, labels=labels) in train mode, then
 * loss.backward() and torch.optim.AdamW over model.parameters().  The reference's training script is
 * not part of the reference tree, so this is the library's contract, pinned by an fp32 autograd
 * restatement (oracle/bart_train_oracle.py).
 *   encoder input  input_ids int32[B, T_enc] ([CLS] hyp [SEP], right-padded), n_valid int32[B] (prefix
 *                  mask): self-attention and cross-attention keys >= n_valid are masked; padded query
 *                  rows are computed.
 *   labels         int32[B, T_dec]; -100 = ignored.
 *   decoder input  shift_tokens_right(labels, pad_id, decoder_start_id): position 0 holds the start id,
 *                  -100 becomes pad_id.  Built inside the library.  Decoder self-attention is causal only
 *                  (no decoder padding mask).
 *   embeddings     LN(shared[id] * embed_scale + embed_positions[i + 2]) then dropout, both stacks.
 *   loss           CrossEntropyLoss() of h . shared^T + final_logits_bias at every decoder position: the
 *                  mean over the positions whose label is not -100.
 *   gradients      shared gets the LM head's part, then the decoder lookup's, then the encoder lookup's
 *                  (the lookups carry embed_scale and send nothing to the pad_id row).  final_logits_bias
 *                  is a buffer: no gradient, no update.  Position rows 0 and 1 get no gradient but are
 *                  decayed by AdamW, like every parameter.
 *   dropout        `dropout` after each embedding LayerNorm, each attention / cross-attention output and
 *                  fc2; `attention_dropout` on the self, causal and cross probabilities.  Stateless hash
 *                  as in pllb_train_*; parity with torch is defined at dropout 0.
 * bf16 GEMM operands, fp32 master weights / gradients / moments, fp32 residual stream, LayerNorm and
 * softmax.  Training takes operand_dtype 0 only; the exported fp32 weights feed pllb_s2s_create with
 * either operand type.  A step is bit-deterministic. */
typedef struct pllb_s2s_train_desc {
  float lr;
  float beta1, beta2;         /* torch.optim.AdamW defaults 0.9, 0.999                              */
  float adam_eps;             /* 1e-8                                                                */
  float weight_decay;         /* applied to every parameter                                          */
  float dropout;              /* BartConfig.dropout (0.1); 0 for parity runs                          */
  float attention_dropout;    /* BartConfig.attention_dropout                                         */
  uint64_t seed;              /* dropout stream                                                       */
  int32_t pad_id;             /* BartConfig.pad_token_id: lookup padding_idx and shifted -100         */
  int32_t decoder_start_id;   /* BartConfig.decoder_start_token_id                                    */
  int32_t max_batch;          /* capacity: sentences per batch                                        */
  int32_t max_enc_len;        /* capacity: T_enc, <= min(enc_max_position, 1024)                      */
  int32_t max_dec_len;        /* capacity: T_dec, <= min(dec_max_position, 1024)                      */
} pllb_s2s_train_desc;

/* desc / weights as pllb_s2s_create, except that enc.pos_emb and dec_pos_emb point at the WHOLE
 * embed_positions tables (max_position + 2 rows: rows 0 and 1 are parameters too) and every pointer,
 * final_logits_bias included, is required.  operand_dtype must be 0 (PLLB_ERR_INVALID otherwise).
 * The handle works with pllb_train_destroy, _reset_optimizer, _workspace_bytes, _kernel_launches,
 * _graph_replays and _row_losses_host; the MLM and RescoreBert calls reject it (PLLB_ERR_INVALID), and
 * the pllb_s2s_train_* calls reject their handles. */
int pllb_s2s_train_create(pllb_trainer* out, const pllb_s2s_desc* desc, const pllb_s2s_weights* weights,
                          const pllb_s2s_train_desc* train, int device);
/* One batch, HOST buffers: input_ids int32[B * T_enc], n_valid int32[B], labels int32[B * T_dec].
 * mode as in pllb_train_step_host (0 loss only, no dropout; 1 update; 2 gradients, no update).
 * PLLB_ERR_INVALID: an id or label outside [0, vocab) other than label -100, n_valid outside [1, T_enc],
 * no label other than -100.  PLLB_ERR_TOO_LONG: T_enc or T_dec above its position table.
 * PLLB_ERR_OOM: B, T_enc or T_dec above the capacity given at create.  One CUDA graph per
 * (B, T_enc, T_dec, mode).  out_loss: the batch loss.  Synchronises.  pllb_train_row_losses_host then
 * returns the B * T_dec per-position losses, 0 where the label is -100. */
int pllb_s2s_train_step_host(pllb_trainer t, const int32_t* input_ids, const int32_t* n_valid, const int32_t* labels,
                             int32_t B, int32_t T_enc, int32_t T_dec, int32_t mode, float* out_loss);
/* The fp32 master weights / the gradients of the last mode-1/2 step into the caller's DEVICE tensors
 * (layout of pllb_s2s_train_create; a NULL pointer skips a tensor).  final_logits_bias: the given
 * values (export) or zeros (export_grads). */
int pllb_s2s_train_export(pllb_trainer t, const pllb_s2s_weights* dst);
int pllb_s2s_train_export_grads(pllb_trainer t, const pllb_s2s_weights* dst);

#ifdef __cplusplus
}
#endif
#endif  /* PLLB_H_ */
