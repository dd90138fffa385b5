// common.h — host-side helpers shared by the translation units of libpllb200.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstdio>
#include <string>
#include <utility>
#include <vector>

#include "../../include/pllb.h"

namespace pllb {

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);
extern thread_local int64_t g_launch_counter;   // kernels launched by this library on this thread
// PLLB_ERR_INVALID unless the kernels support the model shape (scoring and training).  Hidden: library-internal,
// so it does not join the exported symbols.
__attribute__((visibility("hidden"))) int check_model_shape(const pllb_model_desc& d);
// The device check of every create: PLLB_ERR_NO_DEVICE unless an sm_100 device is visible and `device` is sm_100.
// Makes `device` current.
__attribute__((visibility("hidden"))) int check_create_device(int device);

#define PLLB_CUDA(expr)                                                                        \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return ::pllb::fail(PLLB_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));  \
  } while (0)

// returns the error code of a library call that failed
#define RC(expr)            \
  do {                      \
    int _rc = (expr);       \
    if (_rc) return _rc;    \
  } while (0)

// cudaMalloc of max(count, 1) elements, zeroed when asked, recorded in the handle's owned / owned_bytes (its destroy
// frees them; owned_bytes is what the workspace_bytes calls report).
template <typename Ctx, typename T>
int owned_alloc(Ctx* c, T** out, int64_t count, bool zero = false) {
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

#define PLLB_LAUNCH_CHECK(name)                                                                \
  do {                                                                                         \
    ++::pllb::g_launch_counter;                                                                \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess)                                                                     \
      return ::pllb::fail(PLLB_ERR_CUDA, std::string("launch ") + name + ": " + cudaGetErrorString(_e)); \
  } while (0)

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

int sm_count();   // SMs of the current device (cached)

// 2-D row-major tensor [rows, cols] of `elt_bytes`-byte elements, box = [box_rows, box_cols] with
// 128-byte swizzle (box_cols * elt_bytes must be 128).  Encoded once per distinct
// (base, shape, box) and cached per host thread (api.cu).
int get_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int elt_bytes, uint64_t rows, uint64_t cols,
                uint32_t box_rows, uint32_t box_cols);

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per kernel (keyed by its address — every
// instantiation with the same signature has the same pointer TYPE) and device.
template <typename K>
inline cudaError_t opt_in_smem(K kern, int bytes) {
  static thread_local std::vector<std::pair<const void*, int>> done;
  int dev = 0;
  cudaGetDevice(&dev);
  const void* key = reinterpret_cast<const void*>(kern);
  for (const auto& d : done)
    if (d.first == key && d.second == dev) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done.emplace_back(key, dev);
  return e;
}

// ---- GEMM (gemm_tcgen05.cu) -------------------------------------------------
enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,       // out 16-bit = acc + bias
  EPI_BIAS_GELU_BF16 = 1,  // out 16-bit = gelu_erf(acc + bias)
  EPI_BIAS_F32 = 2,        // out fp32 = acc + bias
  EPI_BIAS_GELU_F32 = 3,   // out fp32 = gelu_erf(acc + bias)
  EPI_LSE = 4,             // vocab-tiled online logsumexp + label-column pick (no C output)
  EPI_ARGMAX = 5,          // vocab-tiled (max, first argmax) + label-column pick (no C output); LseArgs.partials
                           // hold (max, __int_as_float(column)) per 128-column half tile
  EPI_TOPK8 = 6,           // beam search (no C output, labels unused): LseArgs.partials hold the EPI_LSE pairs
  EPI_TOPK16 = 7           // [M, 2 * n_tiles_n], then the KSEL (8 / 16) largest (logit, __int_as_float(column))
                           // of every half tile, [M, 2 * n_tiles_n, KSEL], descending, ties to the lower column
};

// Operand-type bits of a GEMM launch:
//   bit 0: A (activations) is IEEE fp16, else bf16      bit 1: W (weights) is fp16, else bf16
//   bit 2: the 16-bit output is written as fp16, else bf16
// tcgen05 kind::f16 encodes the A and B formats in separate descriptor fields, but a launch
// with A = bf16, B = fp16 dies with "illegal instruction" on B200 (measured, round 2): the two
// operands must have the same type, so only the combinations below are instantiated.
enum GemmDtype : int {
  DT_BF16 = 0,          // bf16 x bf16 -> bf16 out
  DT_BF16_OUT16 = 4,    // bf16 x bf16 -> fp16 out (gemm_ln only: feeds the fp16 MLM head of operand mode 2)
  DT_FP16 = 7           // fp16 x fp16 -> fp16 out
};

struct LseArgs {
  const int32_t* labels;   // [M] label column of each row
  float2* partials;        // [M, 2 * n_tiles_n] (running max, sum of exp) per 128-column half tile
  float* label_logit;      // [M] written by the tile that owns the label column
  int32_t vocab;           // real vocab size (columns >= vocab are masked)
};

// C[M,N] = A[M,K] * W[N,K]^T (+ epilogue).  A, W bf16 row-major (K contiguous).
// N % 256 == 0 (pad W rows with zeros), K % 64 == 0.  ldc = N.
// dt: DT_BF16 or DT_FP16.
int launch_gemm_tcgen05(const void* A, const void* W, const float* bias, void* C, int64_t M, int N, int K,
                        int epilogue, const LseArgs* lse, int dt, cudaStream_t stream);
// hidden_f32 = LayerNorm(A * W^T + bias + hidden_f32) in place, hidden_16 = 16-bit copy
// (gemm_ln_tcgen05.cu: cluster of H/256 CTAs per 128-row block, row statistics through DSMEM).
int launch_gemm_ln(const void* A, const void* W, const float* bias, const float* gamma, const float* beta, float eps,
                   float* hidden_f32, void* hidden_16, int64_t M, int H, int K, int dt, cudaStream_t stream);
int launch_gemm_simt(const void* A, const void* W, const float* bias, void* C, int64_t M, int N, int K,
                     int epilogue, cudaStream_t stream);

// ---- fp32 residual stream layout ("T32") ----------------------------------------
// The fp32 hidden states are private to this library, so they are stored in the layout the
// fused GEMM+LayerNorm epilogue wants: rows in blocks of 32; inside a block the 16-byte
// groups of 4 columns of the 32 rows are contiguous:
//     float index of (row, col) = ((row/32 * H/4 + col/4) * 32 + row%32) * 4 + col%4
// A thread that owns one row (the TMEM register layout) then reads / writes consecutive
// 16-byte pieces together with its 31 warp neighbours: 512 contiguous bytes per access.
// Buffers are padded to a multiple of 32 rows.  The 16-bit operand copies stay row-major
// (they are TMA-loaded as GEMM A operands).
__host__ __device__ inline size_t t32_index(int64_t row, int col, int H) {
  return (((size_t)(row >> 5) * (size_t)(H >> 2) + (size_t)(col >> 2)) * 32 + (size_t)(row & 31)) * 4 + (size_t)(col & 3);
}

// ---- encoder pieces (encoder_kernels.cu) -------------------------------------
struct CopyPlan {          // device arrays, one entry per masked copy of the chunk
  int32_t* seq_start;      // first packed row of the copy
  int32_t* seq_len;        // T = L + 2
  int32_t* mask_row;       // packed row index of the [MASK] token
  int32_t* label;          // original token at the masked position
  int32_t* hyp;            // chunk-local hypothesis index
  int32_t* uniq_base;      // first unique row of the copy's hypothesis (layer-0 sharing)
  int32_t* row_src;        // [packed rows] unique row every packed row equals (layer-0 sharing)
};

int launch_expand_plan(const int32_t* tokens, const int32_t* hyp_tok_off, const int32_t* hyp_copy_base,
                       const int32_t* hyp_row_base, int32_t n_hyp, int32_t vocab, bool whole_sequence, CopyPlan plan,
                       cudaStream_t s);
int launch_expand_ids(const int32_t* tokens, const int32_t* hyp_tok_off, CopyPlan plan, int32_t n_copies,
                      int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t* out_ids, int32_t* out_mask_pos,
                      int32_t* out_labels, cudaStream_t s);
int launch_embed_ln(const int32_t* tokens, const int32_t* hyp_tok_off, CopyPlan plan, int32_t n_copies,
                    const float* word_emb, const float* pos_emb, const float* type_emb, const float* g,
                    const float* b, float eps, int H, int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t vocab,
                    float* hidden_f32_rowmajor, void* hidden_bf16, bool fp16, cudaStream_t s);
// out_bf16 = bf16(LN(x)); no residual (MLM head transform)
int launch_plain_ln_bf16(const float* x, void* out_bf16, const float* g, const float* b, float eps, int64_t rows,
                         int H, bool fp16, cudaStream_t s);
// shared_rows: qkv holds the unique rows of every hypothesis (2L+2 per hypothesis) instead of one row per packed row
int launch_attention(const void* qkv_bf16, void* ctx_bf16, CopyPlan plan, int32_t n_copies, int H, int NH, bool fp16,
                     bool shared_rows, cudaStream_t s);
// Embeddings of the unique rows of every hypothesis (fp32 row-major + 16-bit), and the packed-row -> unique-row map.
int launch_embed_unique(const int32_t* tokens, const int32_t* hyp_tok_off, int32_t n_hyp, const float* word_emb,
                        const float* pos_emb, const float* type_emb, const float* g, const float* b, float eps, int H,
                        int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t vocab, float* u_f32, void* u_bf16,
                        bool fp16, cudaStream_t s);
int launch_row_src(CopyPlan plan, int32_t n_copies, cudaStream_t s);
// last layer: one query row per copy (q [copies,H]) against the K|V projection of the whole sequence (kv [rows,2H])
int launch_attention_row(const void* q_bf16, const void* kv_bf16, void* out_bf16, CopyPlan plan, int32_t n_copies, int H,
                         int NH, int max_T, bool fp16, cudaStream_t s);
int launch_gather_rows_bf16(const void* hidden_bf16, const int32_t* rows, int32_t n, int H, void* out,
                            cudaStream_t s);
int launch_gather_rows_f32(const float* src, const int32_t* rows, int32_t n, int H, float* out, cudaStream_t s);
int launch_cls_linear(const float* hid_t32, const float* w, float b, int32_t n, int H, float* out, cudaStream_t s);
int launch_lse_finish(const float2* partials, const float* label_logit, int32_t n_copies, int n_tiles,
                      float* tok_logp, cudaStream_t s);
int launch_hyp_sum(const float* tok_logp, const int32_t* hyp_copy_base, int32_t n_hyp, double* out_pll,
                   float* out_tok_logp, cudaStream_t s);
// T32 blocked fp32 [rows, H] -> row-major fp32 (debug / parity output)
// row_src (optional): packed row r is read from src row row_src[r]
int launch_rowmajor_to_t32(const float* src, const int32_t* row_src, float* dst, int64_t rows, int H, cudaStream_t s);
int launch_t32_to_rowmajor(const float* src, float* dst, int64_t rows, int H, cudaStream_t s);
int launch_f32_to_bf16(const float* src, void* dst, int64_t n, bool fp16, cudaStream_t s);

// ---- combiner (rescore_kernels.cu, compiled with -fmad=false) ------------------
int launch_rescore_sweep(const double* am, const double* lm, const int64_t* len, const int32_t* dist, int32_t N,
                         int32_t n_best, const double* weights, int32_t W, int32_t variant, int32_t* out_argmax,
                         int64_t* out_edit_sum, cudaStream_t s);
int launch_rescore_scores(const double* am, const double* lm, const int64_t* len, int32_t N, int32_t n_best,
                          double weight, int32_t variant, double* out, cudaStream_t s);
int launch_tokenize_count(const int32_t* table, int table_size, const int32_t* cp, const int64_t* cp_off, int32_t n_hyp,
                          int32_t* counts, uint8_t* needs_host, cudaStream_t s);
int launch_tokenize_write(const int32_t* table, int table_size, const int32_t* cp, const int64_t* cp_off, int32_t n_hyp,
                          const uint8_t* needs_host, const int64_t* out_off, int32_t* out_ids, cudaStream_t s);
int launch_levenshtein(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
                       const int32_t* pair_ref, int32_t n_pairs, int32_t max_len, int32_t* out, cudaStream_t s);
// Edit-operation alignment (pllb_align).  align_shape gives the warps of the launch and the
// uint2 words of each warp's global code slot (0: every pair fits the shared-memory codes);
// gcodes must then hold warps * slot_words words.
void align_shape(int32_t n_pairs, int32_t max_ref, int32_t max_hyp, int32_t* warps, int64_t* slot_words);
int launch_align(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
                 const int32_t* pair_ref, int32_t n_pairs, int32_t max_ref, int32_t max_hyp, const int64_t* ops_off,
                 uint8_t* out_ops, int32_t* out_n_ops, int32_t* out_counts, uint2* gcodes, cudaStream_t s);

// ---- BERTScore recall (bertscore_kernels.cu) ------------------------------------------
// out[p] = R(cand, ref) of every pair; pairs come in candidate groups (grp_pair / grp_cand), the
// interior reference rows of pair p are items item_off[p] .. item_off[p+1].  Rows of emb are
// [row_begin, row_end); inv_norm holds row_end - row_begin floats.  One cooperative launch.
int launch_bertscore(const float* emb, const int32_t* row_off, const int32_t* pair_ref, const int32_t* item_off,
                     const int32_t* grp_pair, const int32_t* grp_cand, int32_t n_groups, int H, int32_t row_begin,
                     int32_t row_end, float* inv_norm, float* out, cudaStream_t s);

// ---- greedy seq2seq decoding (seq2seq_kernels.cu) ---------------------------------------
// ids / logit: [rows, max_len] row-major.  done_rows: rows that have emitted EOS (integer counter).
struct DecodeState {
  int32_t* ids;            // [rows, max_len] output ids (position 0 = start token)
  float* logit;            // [rows, max_len] fp32 logit of each chosen token (0 at start / pad positions), or null
  int32_t* len;            // [rows] 0 while unfinished, else the generated length incl. start and EOS
  int32_t* force_col;      // [rows] column whose logit the next head launch picks (forced token) or -1
  int32_t* done_rows;      // [1]
  int32_t rows, max_len, start_id, eos_id, pad_id, forced_bos, forced_eos;   // forced_*: -1 = none
};
int launch_decode_init(DecodeState st, cudaStream_t s);
// hid_f32 (T32) / hid_16 (row-major) = LayerNorm(word_scaled[ids[:, pos]] + pos_emb[pos])
int launch_dec_embed(const DecodeState& st, int pos, const float* word_scaled, const float* pos_emb, const float* g,
                     const float* b, float eps, int H, float* hid_f32, void* hid_16, bool fp16, cudaStream_t s);
// One query row per (row, head) against n keys of that row.  Self form (key_start == null): keys are the
// slots 0..t of the row's cache [rows, max_len, 2H] (K | V); the K | V of slot t are first copied there
// from new_kv ([rows, new_kv_stride], K at column 0, V at H).  Cross form: keys are rows
// key_start[r] .. + key_len[r] of kv (row stride kv_stride, K at column 0, V at H).
// slot (beam search, self form only): key j < self_t of row r is cache row slot[r * max_len + j] of
// the [rows * max_len, 2H] cache instead of row r * max_len + j; key self_t is always the row's own.
int launch_decode_attention(const void* q, int q_stride, const void* kv, int64_t kv_stride, const int32_t* key_start,
                            const int32_t* key_len, int self_t, int max_len, const void* new_kv, int new_kv_stride,
                            void* kv_cache, void* ctx, int rows, int H, int max_keys, bool fp16, cudaStream_t s,
                            const int32_t* slot = nullptr);
// Step t's choice from the EPI_ARGMAX partials: first maximum, forced BOS / EOS, pad after EOS.
int launch_argmax_finish(const float2* partials, const float* forced_logit, int n_parts, DecodeState st, int t,
                         cudaStream_t s);
int launch_scale_copy(const float* src, float* dst, int64_t n, float scale, cudaStream_t s);

// ---- beam search (seq2seq_kernels.cu, DESIGN.md §3.12) ------------------------------------
// A chunk of n sentences decodes n * K beam rows; beam b of sentence i is row i * K + b.  Per row
// [rows, max_len] int32 buffers: running ids and the KV slot table (ping-pong, gathered by parent).
// Per sentence: K finished slots (ids [n * K, max_len], len, score, flag) and the flags below.
struct BeamState {
  int32_t* ids_cur;        // running ids, positions 0 .. t - 1 valid
  int32_t* ids_next;
  int32_t* slot_cur;       // KV slot table, entries 0 .. t - 2 valid
  int32_t* slot_next;
  float* run_score;        // [rows] running beam scores (read, then rewritten in place)
  int32_t* parent;         // [rows] parent row of this step's running beams (chunk-local row index)
  int32_t* fin_ids;        // [rows, max_len]
  int32_t* fin_len;        // [rows]
  float* fin_score;        // [rows]
  int32_t* fin_flag;       // [rows]
  int32_t* sent_flags;     // [n]: bit 0 early-stop heuristic satisfied, bit 1 frozen
  int32_t* frozen_count;   // [1] sentences frozen so far (integer atomic)
  int32_t n, K, max_len, start_id, eos_id, pad_id, forced_bos, forced_eos, early_stopping;   // 0 False 1 True 2 never
  float length_penalty;
};
int launch_beam_init(BeamState st, cudaStream_t s);
// Step t: merge each row's EPI_TOPK partials (n_parts = 2 * vocab tiles of ksel entries each) into its
// log-softmax and top 2K, then apply the beam-search bookkeeping of DESIGN.md §3.12; one CTA per sentence.
int launch_beam_select(const float2* partials, int n_parts, int ksel, int vocab, BeamState st, int t, cudaStream_t s);
// The best r slots of every sentence: ids [n, r, max_len] (pad after the end), len [n, r], score [n, r].
int launch_beam_output(BeamState st, int r, int32_t* out_ids, int32_t* out_len, float* out_score, cudaStream_t s);

}  // namespace pllb
