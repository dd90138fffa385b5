// api.cu — the C ABI of libpllb200.so (include/pllb.h): handle, weight conversion,
// chunked PLL scoring pipeline, host-buffer wrappers and parity/debug hooks.
#include <cuda_bf16.h>

#include <nvtx3/nvToolsExt.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <unordered_map>
#include <vector>

#include "common.h"

namespace pllb {

static thread_local std::string g_last_error;
thread_local int64_t g_launch_counter = 0;

void set_error(const std::string& msg) { g_last_error = msg; }
int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}

int check_model_shape(const pllb_model_desc& d) {
  if (d.hidden % 256 != 0 || d.hidden < 256 || d.hidden > 1024 || d.num_heads * 64 != d.hidden ||
      d.intermediate % 256 != 0 || d.num_layers < 1 || d.vocab < 1 || d.max_position < 3)
    return fail(PLLB_ERR_INVALID, "unsupported model shape: need num_layers >= 1, hidden in {256,512,768,1024}, "
                                  "head dim 64, intermediate % 256 == 0");
  return PLLB_OK;
}

int sm_count() {
  static thread_local int cached_dev = -1, cached = 0;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != cached_dev) {
    cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
    cached_dev = dev;
  }
  return cached;
}

// ---- cached tensor maps --------------------------------------------------------------
// A CUtensorMap depends only on (base, dtype, element size, rows, cols, box): a scoring pass
// re-launches the same handful of shapes on the same workspace buffers for every layer of every
// chunk, so the ~900 cuTensorMapEncodeTiled calls of a C2 step collapse into a few dozen.
namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
struct TmapKey {
  const void* base;
  uint64_t rows, cols;
  uint32_t box_rows, box_cols, dt_elt;
  bool operator==(const TmapKey& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && box_rows == o.box_rows && box_cols == o.box_cols &&
           dt_elt == o.dt_elt;
  }
};
struct TmapHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uint64_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= (k.rows + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (k.cols * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
    h ^= (((uint64_t)k.box_rows << 40) | ((uint64_t)k.box_cols << 16) | k.dt_elt) + (h << 6) + (h >> 2);
    return (size_t)h;
  }
};
thread_local std::unordered_map<TmapKey, CUtensorMap, TmapHash> g_tmaps;
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      return reinterpret_cast<EncodeTiledFn>(p);
    return (EncodeTiledFn) nullptr;
  }();
  return fn;
}
}  // namespace

int get_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dt, int elt_bytes, uint64_t rows, uint64_t cols,
                uint32_t box_rows, uint32_t box_cols) {
  const TmapKey key{base, rows, cols, box_rows, box_cols, ((uint32_t)dt << 8) | (uint32_t)elt_bytes};
  auto it = g_tmaps.find(key);
  if (it != g_tmaps.end()) {
    *out = it->second;
    return PLLB_OK;
  }
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return fail(PLLB_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * (uint64_t)elt_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(PLLB_ERR_CUDA, "cuTensorMapEncodeTiled failed, CUresult " + std::to_string((int)r));
  if (g_tmaps.size() >= 4096) g_tmaps.clear();
  g_tmaps.emplace(key, *out);
  return PLLB_OK;
}

}  // namespace pllb

using namespace pllb;

namespace {

enum GemmKind { G_QKV = 0, G_AO, G_FF1, G_FF2, G_HEAD, G_DEC, G_KINDS };

struct LayerDev {
  __nv_bfloat16 *qkv_w, *ao_w, *ff1_w, *ff2_w;
  float *qkv_b, *ao_b, *ao_g, *ao_be, *ff1_b, *ff2_b, *out_g, *out_be;
};

struct ClsHead {        // Linear(H, 1) applied to the [CLS] state (device pointers)
  const float* w;
  float b;
  float* out;
};

// NVTX range (visible in nsys / ncu --nvtx; a no-op without a tool attached)
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  void next(const char* name) { nvtxRangePop(); nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

struct TimedLaunch {
  cudaEvent_t start, stop;
  int kind;
};

}  // namespace

struct pllb_context {
  pllb_model_desc d{};
  int device = 0;
  // operand types (pllb_model_desc.operand_dtype): encoder layers l < fp16_from work on bf16
  // activations and weights, layers l >= fp16_from on IEEE fp16; the MLM head is fp16 unless the
  // whole model is bf16.  0 bf16 (fp16_from = NL, bf16 head) | 1 fp16 (0) | 2 bf16 encoder + fp16 head
  // (NL) | 3 bf16 first half + fp16 second half and head (NL / 2) | 16 + k (k).
  int fp16_from = 0;
  bool head_fp16 = false;            // the MLM head's activations and weights (transform, decoder) are fp16
  int dt_head = DT_BF16;             // GemmDtype of the head transform + decoder
  bool lfp16(int l) const { return l >= fp16_from; }                       // layer l's 16-bit type is fp16
  int ldt(int l) const { return lfp16(l) ? DT_FP16 : DT_BF16; }            // GemmDtype of layer l's GEMMs
  // FFN2 of layer l writes the 16-bit copy that layer l + 1 (or the head) consumes: in THAT type
  int ldt_ffn2(int l, bool next_fp16) const { return lfp16(l) ? DT_FP16 : (next_fp16 ? DT_BF16_OUT16 : DT_BF16); }
  bool has_head = false;             // MLM head weights were supplied (PLL scoring available)
  bool share_l0 = true;              // embeddings + layer-0 QKV on the unique rows of a hypothesis (PLLB_SHARE_L0=0 disables)
  int64_t cap_rows = 0, cap_copies = 0, cap_hyps = 0;
  int vocab_pad = 0, tiles_v = 0;
  std::vector<void*> owned;          // every cudaMalloc of this handle
  int64_t owned_bytes = 0;
  // parameters
  float *word_emb = nullptr, *pos_emb = nullptr, *type_emb = nullptr, *emb_g = nullptr, *emb_b = nullptr;
  std::vector<LayerDev> layers;
  __nv_bfloat16 *head_w = nullptr, *dec_w = nullptr;
  float *head_b = nullptr, *head_g = nullptr, *head_be = nullptr, *dec_b = nullptr;
  // activations of one chunk
  float *hidden_f32 = nullptr, *y_f32 = nullptr;
  __nv_bfloat16 *hidden_bf16 = nullptr, *wide = nullptr /* qkv [rows,3H] or ffn [rows,I] */, *ctx = nullptr;
  CopyPlan plan{};
  __nv_bfloat16 *hg = nullptr, *t_bf16 = nullptr;
  float *t_f32 = nullptr, *hid_c = nullptr, *label_logit = nullptr, *tok_logp = nullptr;
  float2* partials = nullptr;
  // per-call hypothesis metadata (grown on demand)
  int32_t* meta_dev = nullptr;
  int32_t* meta_host = nullptr;     // pinned
  int64_t meta_cap = 0;
  cudaEvent_t ev_meta = nullptr;    // recorded after the H2D copy of meta_host: the next call waits on it before refilling
  bool meta_pending = false;
  // pllb_bertscore: inverse row norms of the last call (grown on demand, part of the workspace)
  float* bs_norm = nullptr;
  int64_t bs_norm_cap = 0;
  // The workspace (activations, plan, meta_dev) is shared by every call on this handle: each call
  // records ev_done on its stream when it has enqueued everything, and the next call's stream waits
  // on it, so calls issued on different streams are ordered instead of racing on the workspace.
  cudaEvent_t ev_done = nullptr;
  bool done_pending = false;
  // scratch for the _host entry points
  void* io_dev = nullptr;
  int64_t io_cap = 0;
  // stats / timing
  pllb_stats stats{};
  bool timing = false;
  std::vector<TimedLaunch> timed;
  size_t timed_used = 0;
  cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
  bool have_total = false;
  float gemm_ms_kind[G_KINDS] = {0};
  double gemm_flops_kind[G_KINDS] = {0};
};

namespace {

template <typename T>
int dev_alloc(pllb_context* c, T** out, int64_t count) {
  void* p = nullptr;
  const int64_t bytes = std::max<int64_t>(count, 1) * (int64_t)sizeof(T);
  cudaError_t e = cudaMalloc(&p, (size_t)bytes);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(PLLB_ERR_OOM, "cudaMalloc of " + std::to_string(bytes) + " bytes failed: " + cudaGetErrorString(e));
  }
  c->owned.push_back(p);
  c->owned_bytes += bytes;
  *out = reinterpret_cast<T*>(p);
  return PLLB_OK;
}

int copy_f32(pllb_context* c, float** dst, const float* src, int64_t n, cudaStream_t s) {
  int rc = dev_alloc(c, dst, n);
  if (rc) return rc;
  PLLB_CUDA(cudaMemcpyAsync(*dst, src, sizeof(float) * n, cudaMemcpyDeviceToDevice, s));
  return PLLB_OK;
}

int conv_16(pllb_context* c, __nv_bfloat16** dst, const float* src, int64_t n, bool fp16, cudaStream_t s) {
  int rc = dev_alloc(c, dst, n);
  if (rc) return rc;
  return launch_f32_to_bf16(src, *dst, n, fp16, s);
}

#define RC(expr)            \
  do {                      \
    int _rc = (expr);       \
    if (_rc) return _rc;    \
  } while (0)

// Enqueues one GEMM launch (`launch`) on s between the timing events of a timed call, and counts
// its FLOPs towards the stats and its kind.
template <typename Launch>
int timed_launch(pllb_context* c, int kind, double flops, cudaStream_t s, Launch&& launch) {
  TimedLaunch* tl = nullptr;
  if (c->timing) {
    if (c->timed_used == c->timed.size()) {
      TimedLaunch t{};
      PLLB_CUDA(cudaEventCreate(&t.start));
      PLLB_CUDA(cudaEventCreate(&t.stop));
      c->timed.push_back(t);
    }
    tl = &c->timed[c->timed_used++];
    tl->kind = kind;
    PLLB_CUDA(cudaEventRecord(tl->start, s));
  }
  RC(launch());
  if (tl) PLLB_CUDA(cudaEventRecord(tl->stop, s));
  c->stats.gemm_flops += flops;
  c->gemm_flops_kind[kind] += flops;
  c->stats.last_gemm_launches += 1;
  return PLLB_OK;
}

int timed_gemm(pllb_context* c, int kind, const void* A, const void* W, const float* bias, void* C, int64_t M, int N,
               int K, int epi, const LseArgs* lse, cudaStream_t s, int dt) {
  const double fl = 2.0 * (double)M * (double)(epi == EPI_LSE && lse ? lse->vocab : N) * (double)K;
  return timed_launch(c, kind, fl, s, [&] { return launch_gemm_tcgen05(A, W, bias, C, M, N, K, epi, lse, dt, s); });
}

// GEMM + bias + residual + LayerNorm in one kernel (gemm_ln_tcgen05.cu).
int timed_gemm_ln(pllb_context* c, int kind, const void* A, const void* W, const float* bias, const float* g,
                  const float* be, float* hid32, void* hid16, int64_t M, int K, cudaStream_t s, int dt) {
  const int H = c->d.hidden;
  const double fl = 2.0 * (double)M * (double)H * (double)K;
  return timed_launch(c, kind, fl, s,
                      [&] { return launch_gemm_ln(A, W, bias, g, be, c->d.ln_eps, hid32, hid16, M, H, K, dt, s); });
}

// Encoder + head over one chunk whose metadata (tok_off / copy_base / row_base, each
// n_hyp+1 int32) already sits in device memory.  upto_layer < 0: full scoring.
int run_chunk(pllb_context* c, const int32_t* tokens, const int32_t* tok_off, const int32_t* copy_base,
              const int32_t* row_base, int32_t n_hyp, int32_t n_copies, int64_t n_rows, int max_T, double* out_pll,
              float* out_tok_logp, int upto_layer, cudaStream_t s, const ClsHead* cls = nullptr,
              float* out_cls = nullptr) {
  const pllb_model_desc& d = c->d;
  const int H = d.hidden, I = d.intermediate;
  NvtxRange r_chunk("pllb chunk");
  NvtxRange r_stage("stage1: masked-copy expansion + embeddings");
  RC(launch_expand_plan(tokens, tok_off, copy_base, row_base, n_hyp, d.vocab, cls != nullptr, c->plan, s));
  const int n_layers = upto_layer < 0 ? d.num_layers : std::min(upto_layer, d.num_layers);
  // Layer-0 sharing (encoder_kernels.cu, embed_unique_kernel): the masked copies of a hypothesis
  // share all rows but one, and everything up to the layer-0 Q/K/V projection is row-wise, so it
  // runs once per unique row (2L+2 per hypothesis, n_unique in total) instead of once per packed
  // row (L(L+2)).  Bit-identical; used whenever it at least halves the rows.
  const int64_t n_unique = 2 * (int64_t)n_copies + 2 * (int64_t)n_hyp;
  const bool share = c->share_l0 && !cls && 2 * n_unique <= n_rows;
  if (share) {
    // unique embeddings: fp32 row-major in y_f32, 16-bit GEMM operand in ctx (free until attention writes it)
    RC(launch_embed_unique(tokens, tok_off, n_hyp, c->word_emb, c->pos_emb, c->type_emb, c->emb_g, c->emb_b, d.ln_eps,
                           H, d.cls_id, d.sep_id, d.mask_id, d.vocab, c->y_f32, c->ctx, c->lfp16(0), s));
    RC(launch_row_src(c->plan, n_copies, s));
    RC(launch_rowmajor_to_t32(c->y_f32, c->plan.row_src, c->hidden_f32, n_rows, H, s));
  } else {
    RC(launch_embed_ln(tokens, tok_off, c->plan, n_copies, c->word_emb, c->pos_emb, c->type_emb, c->emb_g, c->emb_b,
                       d.ln_eps, H, d.cls_id, d.sep_id, d.mask_id, d.vocab, c->y_f32, c->hidden_bf16, c->lfp16(0), s));
    RC(launch_rowmajor_to_t32(c->y_f32, nullptr, c->hidden_f32, n_rows, H, s));
  }
  // Only the [MASK] row of each copy reaches the MLM head (MLM_PLL/main.py:101), and after the
  // last layer's attention every remaining op is row-wise: the last layer's output
  // projection, LayerNorms and FFN run on the gathered masked rows only (1 row per copy
  // instead of T).  Results are identical; the reference computes and discards the rest.
  const bool prune_last = upto_layer < 0 && n_layers > 0;
  r_stage.next("stage2: encoder");
  for (int l = 0; l < n_layers; ++l) {
    const LayerDev& L = c->layers[l];
    const bool shared_rows = share && l == 0;
    const bool last = prune_last && l == n_layers - 1;
    const bool f16 = c->lfp16(l);            // this layer's activations (hidden16, qkv, ctx, ffn) and weights
    const int dt = c->ldt(l);
    // type of the 16-bit copy this layer's FFN2 leaves behind: the next layer's, or the head's
    const int dt_ffn2 = c->ldt_ffn2(l, l + 1 < d.num_layers ? c->lfp16(l + 1) : (cls ? f16 : c->head_fp16));
    if (last && !shared_rows) {
      // The pruned last layer consumes one attention row per copy: K|V for every row, Q for that
      // row only (1/3 of the projection saved), then a single-query attention straight into hg.
      RC(timed_gemm(c, G_QKV, c->hidden_bf16, L.qkv_w + (size_t)H * H, L.qkv_b + H, c->wide, n_rows, 2 * H, H,
                    EPI_BIAS_BF16, nullptr, s, dt));
      RC(launch_gather_rows_bf16(c->hidden_bf16, c->plan.mask_row, n_copies, H, c->hg, s));
      RC(timed_gemm(c, G_QKV, c->hg, L.qkv_w, L.qkv_b, c->t_bf16, n_copies, H, H, EPI_BIAS_BF16, nullptr, s, dt));
      RC(launch_attention_row(c->t_bf16, c->wide, c->hg, c->plan, n_copies, H, d.num_heads, max_T, f16, s));
    } else {
      RC(timed_gemm(c, G_QKV, shared_rows ? c->ctx : c->hidden_bf16, L.qkv_w, L.qkv_b, c->wide,
                    shared_rows ? n_unique : n_rows, 3 * H, H, EPI_BIAS_BF16, nullptr, s, dt));
      RC(launch_attention(c->wide, c->ctx, c->plan, n_copies, H, d.num_heads, f16, shared_rows, s));
      if (last) RC(launch_gather_rows_bf16(c->ctx, c->plan.mask_row, n_copies, H, c->hg, s));
    }
    if (last) {
      RC(launch_gather_rows_f32(c->hidden_f32, c->plan.mask_row, n_copies, H, c->hid_c, s));
      RC(timed_gemm_ln(c, G_AO, c->hg, L.ao_w, L.ao_b, L.ao_g, L.ao_be, c->hid_c, c->t_bf16, n_copies, H, s, dt));
      RC(timed_gemm(c, G_FF1, c->t_bf16, L.ff1_w, L.ff1_b, c->wide, n_copies, I, H, EPI_BIAS_GELU_BF16, nullptr, s, dt));
      // its 16-bit copy is the MLM head's input: written in the head's operand type
      RC(timed_gemm_ln(c, G_FF2, c->wide, L.ff2_w, L.ff2_b, L.out_g, L.out_be, c->hid_c, c->t_bf16, n_copies, I, s, dt_ffn2));
      break;
    }
    RC(timed_gemm_ln(c, G_AO, c->ctx, L.ao_w, L.ao_b, L.ao_g, L.ao_be, c->hidden_f32, c->hidden_bf16, n_rows, H, s, dt));
    RC(timed_gemm(c, G_FF1, c->hidden_bf16, L.ff1_w, L.ff1_b, c->wide, n_rows, I, H, EPI_BIAS_GELU_BF16, nullptr, s, dt));
    RC(timed_gemm_ln(c, G_FF2, c->wide, L.ff2_w, L.ff2_b, L.out_g, L.out_be, c->hidden_f32, c->hidden_bf16, n_rows, I, s,
                     dt_ffn2));
  }
  if (upto_layer >= 0) return PLLB_OK;
  r_stage.next("stage3: head at the masked rows");
  if (cls) {
    // RescoreBert: lm_score = Linear(H, 1)(last_hidden_state[:, 0, :]) — RescoreBert/model.py:13-21.
    // The pruned last layer left the final [CLS] states in hid_c (fp32, T32 layout).
    if (!prune_last) return fail(PLLB_ERR_INVALID, "sequence scoring needs at least one encoder layer");
    return launch_cls_linear(c->hid_c, cls->w, cls->b, n_copies, H, out_cls, s);
  }
  // MLM head at the masked row of every copy only (the reference evaluates all B*T rows,
  // transformers modeling_bert.py:975, and keeps one: MLM_PLL/main.py:101).
  // (num_layers >= 1, so the pruned last layer always ran and t_bf16 holds the masked rows' final states)
  RC(timed_gemm(c, G_HEAD, c->t_bf16, c->head_w, c->head_b, c->t_f32, n_copies, H, H, EPI_BIAS_GELU_F32, nullptr, s,
                c->dt_head));
  RC(launch_plain_ln_bf16(c->t_f32, c->hg, c->head_g, c->head_be, d.ln_eps, n_copies, H, c->head_fp16, s));
  LseArgs lse{c->plan.label, c->partials, c->label_logit, d.vocab};
  RC(timed_gemm(c, G_DEC, c->hg, c->dec_w, c->dec_b, nullptr, n_copies, c->vocab_pad, H, EPI_LSE, &lse, s, c->dt_head));
  RC(launch_lse_finish(c->partials, c->label_logit, n_copies, 2 * c->tiles_v, c->tok_logp, s));
  RC(launch_hyp_sum(c->tok_logp, copy_base, n_hyp, out_pll, out_tok_logp, s));
  return PLLB_OK;
}

struct Chunk {
  int32_t hyp_begin, n_hyp, n_copies;
  int64_t n_rows, tok_begin;
  int max_T;
  int64_t meta_off;   // offset (in int32) of this chunk's metadata block
};

int ensure_meta(pllb_context* c, int64_t need, cudaStream_t s) {
  if (need <= c->meta_cap) return PLLB_OK;
  PLLB_CUDA(cudaStreamSynchronize(s));
  PLLB_CUDA(cudaDeviceSynchronize());
  if (c->meta_dev) cudaFree(c->meta_dev);
  if (c->meta_host) cudaFreeHost(c->meta_host);
  c->meta_dev = nullptr;
  c->meta_host = nullptr;
  const int64_t cap = need + need / 2 + 1024;
  PLLB_CUDA(cudaMalloc(&c->meta_dev, sizeof(int32_t) * cap));
  PLLB_CUDA(cudaHostAlloc(&c->meta_host, sizeof(int32_t) * cap, cudaHostAllocDefault));
  c->meta_cap = cap;
  return PLLB_OK;
}

// Calls are asynchronous: the previous call's copy out of the pinned metadata buffer may still be
// queued behind its predecessor's kernels.  meta_acquire waits for that copy (not for the
// kernels) before the host refills the buffer; meta_upload copies and records the event.
int meta_acquire(pllb_context* c) {
  if (c->meta_pending) {
    PLLB_CUDA(cudaEventSynchronize(c->ev_meta));
    c->meta_pending = false;
  }
  return PLLB_OK;
}

// Orders this call after the previous one on the same handle (no-op when both use one stream).
int workspace_acquire(pllb_context* c, cudaStream_t s) {
  if (c->done_pending) PLLB_CUDA(cudaStreamWaitEvent(s, c->ev_done, 0));
  return PLLB_OK;
}

int workspace_release(pllb_context* c, cudaStream_t s) {
  if (!c->ev_done) PLLB_CUDA(cudaEventCreateWithFlags(&c->ev_done, cudaEventDisableTiming));
  PLLB_CUDA(cudaEventRecord(c->ev_done, s));
  c->done_pending = true;
  return PLLB_OK;
}

int meta_upload(pllb_context* c, int64_t count, cudaStream_t s) {
  if (count <= 0) return PLLB_OK;
  PLLB_CUDA(cudaMemcpyAsync(c->meta_dev, c->meta_host, sizeof(int32_t) * count, cudaMemcpyHostToDevice, s));
  if (!c->ev_meta) PLLB_CUDA(cudaEventCreateWithFlags(&c->ev_meta, cudaEventDisableTiming));
  PLLB_CUDA(cudaEventRecord(c->ev_meta, s));
  c->meta_pending = true;
  return PLLB_OK;
}

// Plans chunks on the host (offsets are control metadata), uploads the metadata once and
// enqueues every chunk on `s` without synchronising.
// cls != nullptr: sequence-level scoring ([CLS] t [SEP], one pass per hypothesis, Linear(H,1)
// on the [CLS] state) instead of masked-copy PLL scoring; with cls->out == nullptr and
// upto_layer >= 0 only the hidden states of that plan are produced (pllb_embed).
// out_hidden: every chunk's fp32 rows, row-major, at that chunk's first row.
int score_impl(pllb_context* c, const int32_t* hyp_tokens, const int64_t* off, int32_t n_hyp, double* out_pll,
               float* out_tok_logp, int upto_layer, float* out_hidden, cudaStream_t s, const ClsHead* cls = nullptr) {
  if (!c) return fail(PLLB_ERR_INVALID, "null handle");
  if (n_hyp < 0 || (n_hyp > 0 && (!off || !hyp_tokens && off[n_hyp] > off[0])))
    return fail(PLLB_ERR_INVALID, "pllb_score: null argument");
  PLLB_CUDA(cudaSetDevice(c->device));
  const int64_t launches_before = g_launch_counter;
  c->stats.last_gemm_launches = 0;
  c->timed_used = 0;
  std::vector<Chunk> chunks;
  {
    Chunk cur{0, 0, 0, 0, n_hyp > 0 ? off[0] : 0, 0, 0};
    for (int32_t h = 0; h < n_hyp; ++h) {
      const int64_t L = off[h + 1] - off[h];
      if (L < 0) return fail(PLLB_ERR_INVALID, "pllb_score: offsets not monotone");
      if (L + 2 > c->d.max_position)
        return fail(PLLB_ERR_TOO_LONG, "hypothesis " + std::to_string(h) + " has " + std::to_string(L) +
                                           " tokens; max_position_embeddings allows " + std::to_string(c->d.max_position - 2));
      const int64_t rows = cls ? L + 2 : L * (L + 2);
      const int64_t copies = cls ? 1 : L;
      if (rows > c->cap_rows || copies > c->cap_copies)
        return fail(PLLB_ERR_OOM, "a single hypothesis exceeds max_chunk_tokens");
      if (cur.n_hyp > 0 && (cur.n_rows + rows > c->cap_rows || cur.n_copies + copies > c->cap_copies || cur.n_hyp + 1 > c->cap_hyps)) {
        chunks.push_back(cur);
        cur = Chunk{h, 0, 0, 0, off[h], 0, 0};
      }
      cur.n_hyp += 1;
      cur.n_copies += (int32_t)copies;
      cur.n_rows += rows;
      cur.max_T = std::max(cur.max_T, (int)L + 2);
    }
    if (cur.n_hyp > 0) chunks.push_back(cur);
  }
  if (upto_layer >= 0 && !cls && chunks.size() > 1) return fail(PLLB_ERR_OOM, "pllb_debug_hidden: input must fit one chunk");
  int64_t meta_need = 0;
  for (auto& ch : chunks) {
    ch.meta_off = meta_need;
    meta_need += 3 * (int64_t)(ch.n_hyp + 1);
  }
  RC(ensure_meta(c, meta_need, s));
  RC(meta_acquire(c));
  RC(workspace_acquire(c, s));
  for (const auto& ch : chunks) {
    int32_t* tok_off = c->meta_host + ch.meta_off;
    int32_t* copy_base = tok_off + (ch.n_hyp + 1);
    int32_t* row_base = copy_base + (ch.n_hyp + 1);
    int64_t t = 0, cb = 0, rb = 0;
    for (int32_t i = 0; i <= ch.n_hyp; ++i) {
      tok_off[i] = (int32_t)t; copy_base[i] = (int32_t)cb; row_base[i] = (int32_t)rb;
      if (i < ch.n_hyp) {
        const int64_t L = off[ch.hyp_begin + i + 1] - off[ch.hyp_begin + i];
        t += L; cb += cls ? 1 : L; rb += cls ? L + 2 : L * (L + 2);
      }
    }
  }
  RC(meta_upload(c, meta_need, s));
  if (c->timing) {
    if (!c->ev_begin) { PLLB_CUDA(cudaEventCreate(&c->ev_begin)); PLLB_CUDA(cudaEventCreate(&c->ev_end)); }
    PLLB_CUDA(cudaEventRecord(c->ev_begin, s));
  }
  int64_t row0 = 0;
  for (const auto& ch : chunks) {
    const int32_t* tok_off = c->meta_dev + ch.meta_off;
    const int32_t* copy_base = tok_off + (ch.n_hyp + 1);
    const int32_t* row_base = copy_base + (ch.n_hyp + 1);
    RC(run_chunk(c, hyp_tokens + (ch.tok_begin - off[0]), tok_off, copy_base, row_base, ch.n_hyp, ch.n_copies, ch.n_rows,
                 ch.max_T, out_pll ? out_pll + ch.hyp_begin : nullptr,
                 out_tok_logp ? out_tok_logp + (ch.tok_begin - off[0]) : nullptr, upto_layer, s, cls,
                 cls && cls->out ? cls->out + ch.hyp_begin : nullptr));
    if (out_hidden) RC(launch_t32_to_rowmajor(c->hidden_f32, out_hidden + row0 * c->d.hidden, ch.n_rows, c->d.hidden, s));
    row0 += ch.n_rows;
    c->stats.chunks += 1;
    c->stats.hyps_scored += ch.n_hyp;
    c->stats.copies_scored += ch.n_copies;
    c->stats.tokens_expanded += ch.n_rows;
  }
  if (c->timing) { PLLB_CUDA(cudaEventRecord(c->ev_end, s)); c->have_total = true; }
  RC(workspace_release(c, s));
  c->stats.kernel_launches += g_launch_counter - launches_before;
  return PLLB_OK;
}

int ensure_io(pllb_context* c, int64_t bytes) {
  if (bytes <= c->io_cap) return PLLB_OK;
  PLLB_CUDA(cudaDeviceSynchronize());
  if (c->io_dev) cudaFree(c->io_dev);
  c->io_dev = nullptr;
  PLLB_CUDA(cudaMalloc(&c->io_dev, (size_t)(bytes + bytes / 4 + 4096)));
  c->io_cap = bytes + bytes / 4 + 4096;
  return PLLB_OK;
}

int check_device() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(PLLB_ERR_NO_DEVICE, "no CUDA device visible; libpllb200 has no CPU fallback");
  }
  return PLLB_OK;
}

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// Grow-only device scratch for the stage-4 host entry points (one per host thread and
// device): repeated sweeps must not pay cudaMalloc / cudaFree (an implicit device sync).
struct Scratch {
  void* p = nullptr;
  int64_t cap = 0;
  int dev = -1;
};
thread_local Scratch g_scratch;

int get_scratch(int64_t bytes, uint8_t** out) {
  int dev = 0;
  PLLB_CUDA(cudaGetDevice(&dev));
  if (g_scratch.dev != dev || g_scratch.cap < bytes) {
    if (g_scratch.p) {
      PLLB_CUDA(cudaDeviceSynchronize());
      cudaFree(g_scratch.p);
      g_scratch = Scratch{};
    }
    const int64_t cap = bytes + bytes / 2 + (1 << 20);
    PLLB_CUDA(cudaMalloc(&g_scratch.p, (size_t)cap));
    g_scratch.cap = cap;
    g_scratch.dev = dev;
  }
  *out = reinterpret_cast<uint8_t*>(g_scratch.p);
  return PLLB_OK;
}

}  // namespace

extern "C" {

const char* pllb_last_error(void) { return g_last_error.c_str(); }
int pllb_abi_version(void) { return PLLB_ABI_VERSION; }

int pllb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int ok = 0;
  for (int i = 0; i < n; ++i) {
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ++ok;
  }
  return ok;
}

int pllb_create(pllb_handle* out, const pllb_model_desc* desc, const pllb_weights* w, int64_t max_chunk_tokens,
                int device) {
  if (!out || !desc || !w || !w->layers) return fail(PLLB_ERR_INVALID, "pllb_create: null argument");
  *out = nullptr;
  RC(check_device());
  const pllb_model_desc& d = *desc;
  RC(check_model_shape(d));
  if (d.operand_dtype < 0 || (d.operand_dtype > 3 && (d.operand_dtype < 16 || d.operand_dtype > 16 + d.num_layers)))
    return fail(PLLB_ERR_INVALID, "unsupported model shape: need num_layers >= 1, hidden in {256,512,768,1024}, "
                                  "head dim 64, intermediate % 256 == 0");
  PLLB_CUDA(cudaSetDevice(device));
  int major = 0;
  PLLB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(PLLB_ERR_NO_DEVICE, "device is not sm_100 (B200); libpllb200 has no other code path");
  pllb_context* c = new pllb_context();
  c->d = d;
  c->device = device;
  c->fp16_from = d.operand_dtype == 1 ? 0 : d.operand_dtype == 3 ? d.num_layers / 2
               : d.operand_dtype >= 16 ? d.operand_dtype - 16 : d.num_layers;
  c->head_fp16 = d.operand_dtype >= 1;
  c->dt_head = c->head_fp16 ? DT_FP16 : DT_BF16;
  if (const char* e = getenv("PLLB_SHARE_L0")) c->share_l0 = atoi(e) != 0;
  cudaStream_t s = 0;
  const int H = d.hidden, I = d.intermediate, V = d.vocab;
  int rc = PLLB_OK;
  auto bail = [&](int code) {
    pllb_destroy(c);
    return code;
  };
#define TRY(expr)                  \
  do {                             \
    rc = (expr);                   \
    if (rc) return bail(rc);       \
  } while (0)
  TRY(copy_f32(c, &c->word_emb, w->word_emb, (int64_t)V * H, s));
  TRY(copy_f32(c, &c->pos_emb, w->pos_emb, (int64_t)d.max_position * H, s));
  TRY(copy_f32(c, &c->type_emb, w->type_emb, H, s));   // token_type 0 only (MLM_PLL/main.py:89-94 passes none)
  TRY(copy_f32(c, &c->emb_g, w->emb_ln_g, H, s));
  TRY(copy_f32(c, &c->emb_b, w->emb_ln_b, H, s));
  c->layers.resize(d.num_layers);
  for (int l = 0; l < d.num_layers; ++l) {
    const pllb_layer_weights& lw = w->layers[l];
    LayerDev& L = c->layers[l];
    TRY(dev_alloc(c, &L.qkv_w, (int64_t)3 * H * H));
    TRY(launch_f32_to_bf16(lw.q_w, L.qkv_w, (int64_t)H * H, c->lfp16(l), s));
    TRY(launch_f32_to_bf16(lw.k_w, L.qkv_w + (int64_t)H * H, (int64_t)H * H, c->lfp16(l), s));
    TRY(launch_f32_to_bf16(lw.v_w, L.qkv_w + (int64_t)2 * H * H, (int64_t)H * H, c->lfp16(l), s));
    TRY(dev_alloc(c, &L.qkv_b, 3 * H));
    cudaMemcpyAsync(L.qkv_b, lw.q_b, sizeof(float) * H, cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(L.qkv_b + H, lw.k_b, sizeof(float) * H, cudaMemcpyDeviceToDevice, s);
    cudaMemcpyAsync(L.qkv_b + 2 * H, lw.v_b, sizeof(float) * H, cudaMemcpyDeviceToDevice, s);
    TRY(conv_16(c, &L.ao_w, lw.ao_w, (int64_t)H * H, c->lfp16(l), s));
    TRY(copy_f32(c, &L.ao_b, lw.ao_b, H, s));
    TRY(copy_f32(c, &L.ao_g, lw.ao_ln_g, H, s));
    TRY(copy_f32(c, &L.ao_be, lw.ao_ln_b, H, s));
    TRY(conv_16(c, &L.ff1_w, lw.ff1_w, (int64_t)I * H, c->lfp16(l), s));
    TRY(copy_f32(c, &L.ff1_b, lw.ff1_b, I, s));
    TRY(conv_16(c, &L.ff2_w, lw.ff2_w, (int64_t)H * I, c->lfp16(l), s));
    TRY(copy_f32(c, &L.ff2_b, lw.ff2_b, H, s));
    TRY(copy_f32(c, &L.out_g, lw.out_ln_g, H, s));
    TRY(copy_f32(c, &L.out_be, lw.out_ln_b, H, s));
  }
  c->vocab_pad = (int)align_up(V, 256);
  c->tiles_v = c->vocab_pad / 256;
  // the MLM head is optional: a RescoreBert checkpoint (BertModel + Linear) has none
  c->has_head = w->head_w && w->head_b && w->head_ln_g && w->head_ln_b && w->decoder_w && w->decoder_b;
  if (c->has_head) {
    TRY(dev_alloc(c, &c->head_w, (int64_t)H * H));
    TRY(launch_f32_to_bf16(w->head_w, c->head_w, (int64_t)H * H, c->head_fp16, s));
    TRY(copy_f32(c, &c->head_b, w->head_b, H, s));
    TRY(copy_f32(c, &c->head_g, w->head_ln_g, H, s));
    TRY(copy_f32(c, &c->head_be, w->head_ln_b, H, s));
    TRY(dev_alloc(c, &c->dec_w, (int64_t)c->vocab_pad * H));
    cudaMemsetAsync(c->dec_w, 0, sizeof(__nv_bfloat16) * (size_t)c->vocab_pad * H, s);
    TRY(launch_f32_to_bf16(w->decoder_w, c->dec_w, (int64_t)V * H, c->head_fp16, s));
    TRY(dev_alloc(c, &c->dec_b, c->vocab_pad));
    cudaMemsetAsync(c->dec_b, 0, sizeof(float) * c->vocab_pad, s);
    cudaMemcpyAsync(c->dec_b, w->decoder_b, sizeof(float) * V, cudaMemcpyDeviceToDevice, s);
  }

  // workspace: sized by the expanded-token budget of one chunk
  if (max_chunk_tokens <= 0) max_chunk_tokens = (int64_t)1 << 20;
  c->cap_rows = align_up(std::max<int64_t>(max_chunk_tokens, 1024), 256);   // the paired LayerNorm clusters work on 256-row blocks
  c->cap_copies = c->cap_rows / 4 + 128;
  c->cap_hyps = c->cap_rows / 4 + 128;
  const int64_t R = c->cap_rows, C = c->cap_copies;
  const int wide = std::max(3 * H, I);
  TRY(dev_alloc(c, &c->hidden_f32, R * H));
  TRY(dev_alloc(c, &c->hidden_bf16, R * H));
  TRY(dev_alloc(c, &c->wide, R * wide));
  TRY(dev_alloc(c, &c->ctx, R * H));
  TRY(dev_alloc(c, &c->y_f32, R * H));
  TRY(dev_alloc(c, &c->plan.seq_start, C));
  TRY(dev_alloc(c, &c->plan.seq_len, C));
  TRY(dev_alloc(c, &c->plan.mask_row, C));
  TRY(dev_alloc(c, &c->plan.label, C));
  TRY(dev_alloc(c, &c->plan.hyp, C));
  TRY(dev_alloc(c, &c->plan.uniq_base, C));
  TRY(dev_alloc(c, &c->plan.row_src, R));
  TRY(dev_alloc(c, &c->hg, C * H));
  TRY(dev_alloc(c, &c->t_f32, C * H));
  TRY(dev_alloc(c, &c->hid_c, align_up(C, 256) * H));
  TRY(dev_alloc(c, &c->t_bf16, C * H));
  TRY(dev_alloc(c, &c->partials, C * c->tiles_v * 2));
  TRY(dev_alloc(c, &c->label_logit, C));
  TRY(dev_alloc(c, &c->tok_logp, C));
#undef TRY
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    pllb_destroy(c);
    return fail(PLLB_ERR_CUDA, std::string("pllb_create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return PLLB_OK;
}

int pllb_destroy(pllb_handle h) {
  if (!h) return PLLB_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (void* p : h->owned) cudaFree(p);
  if (h->meta_dev) cudaFree(h->meta_dev);
  if (h->meta_host) cudaFreeHost(h->meta_host);
  if (h->bs_norm) cudaFree(h->bs_norm);
  if (h->ev_meta) cudaEventDestroy(h->ev_meta);
  if (h->ev_done) cudaEventDestroy(h->ev_done);
  if (h->io_dev) cudaFree(h->io_dev);
  for (auto& t : h->timed) { cudaEventDestroy(t.start); cudaEventDestroy(t.stop); }
  if (h->ev_begin) { cudaEventDestroy(h->ev_begin); cudaEventDestroy(h->ev_end); }
  delete h;
  return PLLB_OK;
}

int64_t pllb_workspace_bytes(pllb_handle h) { return h ? h->owned_bytes : 0; }

int pllb_score(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets, int32_t n_hyp, double* out_pll,
               float* out_token_logp, void* stream) {
  if (!out_pll && n_hyp > 0) return fail(PLLB_ERR_INVALID, "pllb_score: out_pll is null");
  if (h && !h->has_head) return fail(PLLB_ERR_INVALID, "pllb_score: the handle was created without MLM head weights");
  if (n_hyp > 0 && !hyp_offsets) return fail(PLLB_ERR_INVALID, "pllb_score: hyp_offsets is null");
  const int64_t o0 = n_hyp > 0 ? hyp_offsets[0] : 0;   // tokens / token_logp are indexed by absolute offset
  return score_impl(h, hyp_tokens ? hyp_tokens + o0 : nullptr, hyp_offsets, n_hyp, out_pll,
                    out_token_logp ? out_token_logp + o0 : nullptr, -1, nullptr, (cudaStream_t)stream);
}

int pllb_score_host(pllb_handle h, const int32_t* hyp_tokens, const int64_t* off, int32_t n_hyp, double* out_pll,
                    float* out_token_logp) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  if (n_hyp <= 0) return PLLB_OK;
  if (!off || !out_pll) return fail(PLLB_ERR_INVALID, "pllb_score_host: null argument");
  if (!h->has_head) return fail(PLLB_ERR_INVALID, "pllb_score_host: the handle was created without MLM head weights");
  PLLB_CUDA(cudaSetDevice(h->device));
  const int64_t n_tok = off[n_hyp] - off[0];
  if (n_tok > 0 && !hyp_tokens) return fail(PLLB_ERR_INVALID, "pllb_score_host: hyp_tokens is null");
  // the reference's embedding lookup raises IndexError on an id outside the vocabulary
  for (int64_t i = off[0]; i < off[n_hyp]; ++i)
    if (hyp_tokens[i] < 0 || hyp_tokens[i] >= h->d.vocab)
      return fail(PLLB_ERR_INVALID, "token id " + std::to_string(hyp_tokens[i]) + " at position " + std::to_string(i) +
                                        " is outside the vocabulary [0, " + std::to_string(h->d.vocab) + ")");
  const int64_t b_tok = align_up(sizeof(int32_t) * std::max<int64_t>(n_tok, 1), 256);
  const int64_t b_pll = align_up(sizeof(double) * n_hyp, 256);
  const int64_t b_lp = align_up(sizeof(float) * std::max<int64_t>(n_tok, 1), 256);
  RC(ensure_io(h, b_tok + b_pll + b_lp));
  uint8_t* base = reinterpret_cast<uint8_t*>(h->io_dev);
  int32_t* d_tok = reinterpret_cast<int32_t*>(base);
  double* d_pll = reinterpret_cast<double*>(base + b_tok);
  float* d_lp = reinterpret_cast<float*>(base + b_tok + b_pll);
  cudaStream_t s = 0;
  if (n_tok > 0)
    PLLB_CUDA(cudaMemcpyAsync(d_tok, hyp_tokens + off[0], sizeof(int32_t) * n_tok, cudaMemcpyHostToDevice, s));
  RC(score_impl(h, d_tok, off, n_hyp, d_pll, out_token_logp ? d_lp : nullptr, -1, nullptr, s));
  PLLB_CUDA(cudaMemcpyAsync(out_pll, d_pll, sizeof(double) * n_hyp, cudaMemcpyDeviceToHost, s));
  if (out_token_logp && n_tok > 0)
    PLLB_CUDA(cudaMemcpyAsync(out_token_logp + off[0], d_lp, sizeof(float) * n_tok, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  return PLLB_OK;
}

int pllb_score_cls(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets, int32_t n_hyp,
                   const float* linear_w, float linear_b, float* out_scores, void* stream) {
  if (n_hyp > 0 && (!hyp_offsets || !linear_w || !out_scores)) return fail(PLLB_ERR_INVALID, "pllb_score_cls: null argument");
  const int64_t o0 = n_hyp > 0 ? hyp_offsets[0] : 0;
  ClsHead cls{linear_w, linear_b, out_scores};
  return score_impl(h, hyp_tokens ? hyp_tokens + o0 : nullptr, hyp_offsets, n_hyp, nullptr, nullptr, -1, nullptr,
                    (cudaStream_t)stream, &cls);
}

int pllb_score_cls_host(pllb_handle h, const int32_t* hyp_tokens, const int64_t* off, int32_t n_hyp,
                        const float* linear_w, float linear_b, float* out_scores) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  if (n_hyp <= 0) return PLLB_OK;
  if (!off || !linear_w || !out_scores) return fail(PLLB_ERR_INVALID, "pllb_score_cls_host: null argument");
  PLLB_CUDA(cudaSetDevice(h->device));
  const int64_t n_tok = off[n_hyp] - off[0];
  if (n_tok > 0 && !hyp_tokens) return fail(PLLB_ERR_INVALID, "pllb_score_cls_host: hyp_tokens is null");
  for (int64_t i = off[0]; i < off[n_hyp]; ++i)
    if (hyp_tokens[i] < 0 || hyp_tokens[i] >= h->d.vocab)
      return fail(PLLB_ERR_INVALID, "token id " + std::to_string(hyp_tokens[i]) + " is outside the vocabulary");
  const int H = h->d.hidden;
  const int64_t b_tok = align_up(sizeof(int32_t) * std::max<int64_t>(n_tok, 1), 256);
  const int64_t b_out = align_up(sizeof(float) * n_hyp, 256), b_w = align_up(sizeof(float) * H, 256);
  RC(ensure_io(h, b_tok + b_out + b_w));
  uint8_t* base = reinterpret_cast<uint8_t*>(h->io_dev);
  int32_t* d_tok = reinterpret_cast<int32_t*>(base);
  float* d_out = reinterpret_cast<float*>(base + b_tok);
  float* d_w = reinterpret_cast<float*>(base + b_tok + b_out);
  cudaStream_t s = 0;
  if (n_tok > 0) PLLB_CUDA(cudaMemcpyAsync(d_tok, hyp_tokens + off[0], sizeof(int32_t) * n_tok, cudaMemcpyHostToDevice, s));
  PLLB_CUDA(cudaMemcpyAsync(d_w, linear_w, sizeof(float) * H, cudaMemcpyHostToDevice, s));
  ClsHead cls{d_w, linear_b, d_out};
  RC(score_impl(h, d_tok, off, n_hyp, nullptr, nullptr, -1, nullptr, s, &cls));
  PLLB_CUDA(cudaMemcpyAsync(out_scores, d_out, sizeof(float) * n_hyp, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  return PLLB_OK;
}

int pllb_expand(pllb_handle h, const int32_t* hyp_tokens, const int64_t* off, int32_t n_hyp, int32_t* out_ids,
                int32_t* out_mask_pos, int32_t* out_labels, void* stream) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  if (n_hyp <= 0) return PLLB_OK;
  cudaStream_t s = (cudaStream_t)stream;
  PLLB_CUDA(cudaSetDevice(h->device));
  int64_t copies = 0, rows = 0;
  for (int32_t i = 0; i < n_hyp; ++i) {
    const int64_t L = off[i + 1] - off[i];
    copies += L;
    rows += L * (L + 2);
  }
  if (copies > h->cap_copies || rows > INT32_MAX || n_hyp > h->cap_hyps)
    return fail(PLLB_ERR_OOM, "pllb_expand: input exceeds one chunk");
  RC(ensure_meta(h, 3 * (int64_t)(n_hyp + 1), s));
  RC(meta_acquire(h));
  RC(workspace_acquire(h, s));
  int32_t* tok_off = h->meta_host;
  int32_t* copy_base = tok_off + (n_hyp + 1);
  int32_t* row_base = copy_base + (n_hyp + 1);
  int64_t t = 0, cb = 0, rb = 0;
  for (int32_t i = 0; i <= n_hyp; ++i) {
    tok_off[i] = (int32_t)t; copy_base[i] = (int32_t)cb; row_base[i] = (int32_t)rb;
    if (i < n_hyp) { const int64_t L = off[i + 1] - off[i]; t += L; cb += L; rb += L * (L + 2); }
  }
  RC(meta_upload(h, 3 * (int64_t)(n_hyp + 1), s));
  const int32_t* d_tok_off = h->meta_dev;
  hyp_tokens += off[0];
  RC(launch_expand_plan(hyp_tokens, d_tok_off, d_tok_off + (n_hyp + 1), d_tok_off + 2 * (n_hyp + 1), n_hyp, h->d.vocab,
                        false, h->plan, s));
  RC(launch_expand_ids(hyp_tokens, d_tok_off, h->plan, (int32_t)copies, h->d.cls_id, h->d.sep_id, h->d.mask_id, out_ids,
                       out_mask_pos, out_labels, s));
  return workspace_release(h, s);
}

int pllb_get_stats(pllb_handle h, pllb_stats* out) {
  if (!h || !out) return fail(PLLB_ERR_INVALID, "pllb_get_stats: null argument");
  if (h->timing && h->have_total) {
    PLLB_CUDA(cudaEventSynchronize(h->ev_end));
    float total = 0.f, gemm = 0.f;
    PLLB_CUDA(cudaEventElapsedTime(&total, h->ev_begin, h->ev_end));
    for (int k = 0; k < G_KINDS; ++k) h->gemm_ms_kind[k] = 0.f;
    for (size_t i = 0; i < h->timed_used; ++i) {
      float ms = 0.f;
      PLLB_CUDA(cudaEventElapsedTime(&ms, h->timed[i].start, h->timed[i].stop));
      gemm += ms;
      h->gemm_ms_kind[h->timed[i].kind] += ms;
    }
    h->stats.last_total_ms = total;
    h->stats.last_gemm_ms = gemm;
  }
  *out = h->stats;
  return PLLB_OK;
}

/* Per-GEMM-kind device time (ms) of the last timed pllb_score call and the FLOPs issued
 * per kind since the last reset: order QKV, attn-out, FFN1, FFN2, head transform, decoder. */
int pllb_get_gemm_breakdown(pllb_handle h, float* ms6, double* flops6) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  for (int k = 0; k < G_KINDS; ++k) {
    if (ms6) ms6[k] = h->gemm_ms_kind[k];
    if (flops6) flops6[k] = h->gemm_flops_kind[k];
  }
  return PLLB_OK;
}

int pllb_reset_stats(pllb_handle h) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  h->stats = pllb_stats{};
  for (int k = 0; k < G_KINDS; ++k) { h->gemm_ms_kind[k] = 0.f; h->gemm_flops_kind[k] = 0.0; }
  h->have_total = false;
  return PLLB_OK;
}

int pllb_set_timing(pllb_handle h, int enable) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  h->timing = enable != 0;
  return PLLB_OK;
}

int pllb_debug_gemm(const uint16_t* A, const uint16_t* W, const float* bias, void* C, int32_t M, int32_t N, int32_t K,
                    int32_t epilogue, void* stream) {
  RC(check_device());
  if (epilogue < 0 || epilogue > 3) return fail(PLLB_ERR_INVALID, "pllb_debug_gemm: epilogue must be 0..3");
  return launch_gemm_tcgen05(A, W, bias, C, M, N, K, epilogue, nullptr, DT_BF16, (cudaStream_t)stream);
}

int pllb_debug_gemm_dt(const uint16_t* A, const uint16_t* W, const float* bias, void* C, int32_t M, int32_t N, int32_t K,
                       int32_t epilogue, int32_t operand_dtype, void* stream) {
  RC(check_device());
  if (epilogue < 0 || epilogue > 3) return fail(PLLB_ERR_INVALID, "pllb_debug_gemm_dt: epilogue must be 0..3");
  if (operand_dtype < 0 || operand_dtype > 1) return fail(PLLB_ERR_INVALID, "pllb_debug_gemm_dt: operand_dtype must be 0 or 1");
  const int dt = operand_dtype == 1 ? DT_FP16 : DT_BF16;
  return launch_gemm_tcgen05(A, W, bias, C, M, N, K, epilogue, nullptr, dt, (cudaStream_t)stream);
}

int pllb_debug_gemm_simt(const uint16_t* A, const uint16_t* W, const float* bias, void* C, int32_t M, int32_t N,
                         int32_t K, int32_t epilogue, void* stream) {
  RC(check_device());
  return launch_gemm_simt(A, W, bias, C, M, N, K, epilogue, (cudaStream_t)stream);
}

int pllb_debug_hidden(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets, int32_t n_hyp,
                      int32_t upto_layer, float* out_hidden, void* stream) {
  if (upto_layer < 0) return fail(PLLB_ERR_INVALID, "pllb_debug_hidden: upto_layer must be >= 0");
  if (n_hyp > 0 && !hyp_offsets) return fail(PLLB_ERR_INVALID, "pllb_debug_hidden: hyp_offsets is null");
  const int64_t o0 = n_hyp > 0 ? hyp_offsets[0] : 0;
  return score_impl(h, hyp_tokens ? hyp_tokens + o0 : nullptr, hyp_offsets, n_hyp, nullptr, nullptr, upto_layer,
                    out_hidden, (cudaStream_t)stream);
}

int pllb_embed(pllb_handle h, const int32_t* hyp_tokens, const int64_t* hyp_offsets, int32_t n_hyp, int32_t num_layers,
               float* out_hidden, void* stream) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  if (num_layers < 0 || num_layers > h->d.num_layers)
    return fail(PLLB_ERR_INVALID, "pllb_embed: num_layers must be in [0, " + std::to_string(h->d.num_layers) + "]");
  if (n_hyp > 0 && (!hyp_offsets || !out_hidden)) return fail(PLLB_ERR_INVALID, "pllb_embed: null argument");
  const int64_t o0 = n_hyp > 0 ? hyp_offsets[0] : 0;
  ClsHead plan_only{nullptr, 0.f, nullptr};     // the [CLS] t [SEP] plan, no head
  return score_impl(h, hyp_tokens ? hyp_tokens + o0 : nullptr, hyp_offsets, n_hyp, nullptr, nullptr, num_layers,
                    out_hidden, (cudaStream_t)stream, &plan_only);
}

int pllb_bertscore(pllb_handle h, const float* emb, const int64_t* row_off, int32_t n_seq, const int32_t* cand,
                   const int32_t* ref, int32_t n_pairs, float* out_recall, void* stream) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  if (n_seq < 0 || n_pairs < 0) return fail(PLLB_ERR_INVALID, "pllb_bertscore: negative count");
  if (n_pairs == 0) return PLLB_OK;
  if (!emb || !row_off || !cand || !ref || !out_recall) return fail(PLLB_ERR_INVALID, "pllb_bertscore: null argument");
  if (reinterpret_cast<uintptr_t>(emb) % 16 != 0) return fail(PLLB_ERR_INVALID, "pllb_bertscore: emb must be 16-byte aligned");
  if (row_off[0] < 0 || row_off[n_seq] > INT32_MAX) return fail(PLLB_ERR_INVALID, "pllb_bertscore: row offsets out of range");
  for (int32_t i = 0; i < n_seq; ++i)
    if (row_off[i + 1] - row_off[i] < 2)
      return fail(PLLB_ERR_INVALID, "pllb_bertscore: sequence " + std::to_string(i) +
                                        (row_off[i + 1] < row_off[i] ? " has non-monotone row offsets"
                                                                     : " has fewer than 2 rows ([CLS] and [SEP])"));
  // candidate groups: runs of consecutive pairs with the same candidate (one CTA each)
  int64_t items = 0;
  int32_t n_groups = 0;
  for (int32_t p = 0; p < n_pairs; ++p) {
    if (cand[p] < 0 || cand[p] >= n_seq || ref[p] < 0 || ref[p] >= n_seq)
      return fail(PLLB_ERR_INVALID, "pllb_bertscore: pair " + std::to_string(p) + " names a sequence outside [0, " +
                                        std::to_string(n_seq) + ")");
    items += row_off[ref[p] + 1] - row_off[ref[p]] - 2;
    if (p == 0 || cand[p] != cand[p - 1]) ++n_groups;
  }
  if (items > INT32_MAX) return fail(PLLB_ERR_INVALID, "pllb_bertscore: too many reference rows in one call");
  cudaStream_t s = (cudaStream_t)stream;
  PLLB_CUDA(cudaSetDevice(h->device));
  const int64_t n_rows = row_off[n_seq] - row_off[0];
  // metadata (int32): row_off[n_seq+1] | pair_ref[n_pairs] | item_off[n_pairs+1] | grp_pair[n_groups+1] | grp_cand[n_groups]
  const int64_t meta = (int64_t)(n_seq + 1) + n_pairs + (n_pairs + 1) + (n_groups + 1) + n_groups;
  RC(ensure_meta(h, meta, s));
  RC(meta_acquire(h));
  RC(workspace_acquire(h, s));
  if (n_rows > h->bs_norm_cap) {
    PLLB_CUDA(cudaStreamSynchronize(s));
    PLLB_CUDA(cudaDeviceSynchronize());
    if (h->bs_norm) cudaFree(h->bs_norm);
    h->bs_norm = nullptr;
    h->bs_norm_cap = 0;
    const int64_t cap = n_rows + n_rows / 2 + 1024;
    PLLB_CUDA(cudaMalloc(&h->bs_norm, sizeof(float) * cap));
    h->bs_norm_cap = cap;
  }
  int32_t* m_row = h->meta_host;
  int32_t* m_ref = m_row + (n_seq + 1);
  int32_t* m_item = m_ref + n_pairs;
  int32_t* m_gp = m_item + (n_pairs + 1);
  int32_t* m_gc = m_gp + (n_groups + 1);
  for (int32_t i = 0; i <= n_seq; ++i) m_row[i] = (int32_t)row_off[i];
  m_item[0] = 0;
  for (int32_t p = 0, g = 0; p < n_pairs; ++p) {
    m_ref[p] = ref[p];
    m_item[p + 1] = m_item[p] + (int32_t)(row_off[ref[p] + 1] - row_off[ref[p]] - 2);
    if (p == 0 || cand[p] != cand[p - 1]) { m_gp[g] = p; m_gc[g] = cand[p]; ++g; }
  }
  m_gp[n_groups] = n_pairs;
  RC(meta_upload(h, meta, s));
  const int32_t* d = h->meta_dev;
  const int32_t* d_row = d;
  const int32_t* d_ref = d_row + (n_seq + 1);
  const int32_t* d_item = d_ref + n_pairs;
  const int32_t* d_gp = d_item + (n_pairs + 1);
  const int32_t* d_gc = d_gp + (n_groups + 1);
  const int64_t launches_before = g_launch_counter;
  RC(launch_bertscore(emb, d_row, d_ref, d_item, d_gp, d_gc, n_groups, h->d.hidden, (int32_t)row_off[0],
                      (int32_t)row_off[n_seq], h->bs_norm, out_recall, s));
  h->stats.kernel_launches += g_launch_counter - launches_before;
  return workspace_release(h, s);
}

int pllb_levenshtein(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
                     const int32_t* pair_ref, int32_t n_pairs, int32_t max_len, int32_t* out_dist, void* stream) {
  RC(check_device());
  NvtxRange r("stage4: levenshtein");
  return launch_levenshtein(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref, n_pairs, max_len, out_dist, (cudaStream_t)stream);
}

int pllb_tokenize_host(const int32_t* table, int32_t table_size, const int32_t* cp, const int64_t* cp_off, int32_t n_hyp,
                       int32_t* out_ids, int64_t* out_off, uint8_t* needs_host) {
  RC(check_device());
  if (n_hyp < 0 || table_size <= 0) return fail(PLLB_ERR_INVALID, "pllb_tokenize_host: bad size");
  if (!table || !cp_off || !out_off || (n_hyp > 0 && !needs_host)) return fail(PLLB_ERR_INVALID, "pllb_tokenize_host: null argument");
  out_off[0] = 0;
  if (n_hyp == 0) return PLLB_OK;
  const int64_t n_cp = cp_off[n_hyp] - cp_off[0];
  if (n_cp < 0 || (n_cp > 0 && (!cp || !out_ids))) return fail(PLLB_ERR_INVALID, "pllb_tokenize_host: bad offsets");
  for (int32_t i = 0; i < n_hyp; ++i)
    if (cp_off[i + 1] < cp_off[i]) return fail(PLLB_ERR_INVALID, "pllb_tokenize_host: offsets not ascending");
  const int64_t b0 = align_up(4 * (int64_t)table_size, 256), b1 = align_up(4 * std::max<int64_t>(n_cp, 1), 256),
                b2 = align_up(8 * (int64_t)(n_hyp + 1), 256), b3 = align_up(4 * (int64_t)n_hyp, 256),
                b4 = align_up((int64_t)n_hyp, 256), b5 = b2, b6 = b1;
  uint8_t* base = nullptr;
  RC(get_scratch(b0 + b1 + b2 + b3 + b4 + b5 + b6, &base));
  int32_t* d_table = (int32_t*)base;
  int32_t* d_cp = (int32_t*)(base + b0);
  int64_t* d_off = (int64_t*)(base + b0 + b1);
  int32_t* d_cnt = (int32_t*)(base + b0 + b1 + b2);
  uint8_t* d_flag = base + b0 + b1 + b2 + b3;
  int64_t* d_ooff = (int64_t*)(base + b0 + b1 + b2 + b3 + b4);
  int32_t* d_ids = (int32_t*)(base + b0 + b1 + b2 + b3 + b4 + b5);
  cudaStream_t s = 0;
  std::vector<int64_t> rel(n_hyp + 1);                        // offsets relative to the first code point
  for (int32_t i = 0; i <= n_hyp; ++i) rel[i] = cp_off[i] - cp_off[0];
  std::vector<int32_t> cnt(n_hyp);
  int rc = PLLB_OK;
  cudaError_t e = cudaMemcpyAsync(d_table, table, 4 * (int64_t)table_size, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && n_cp > 0) e = cudaMemcpyAsync(d_cp, cp + cp_off[0], 4 * n_cp, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_off, rel.data(), 8 * (int64_t)(n_hyp + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) rc = launch_tokenize_count(d_table, table_size, d_cp, d_off, n_hyp, d_cnt, d_flag, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(cnt.data(), d_cnt, 4 * (int64_t)n_hyp, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(needs_host, d_flag, n_hyp, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaStreamSynchronize(s);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("pllb_tokenize_host: ") + cudaGetErrorString(e));
  for (int32_t i = 0; i < n_hyp; ++i) out_off[i + 1] = out_off[i] + cnt[i];
  const int64_t n_out = out_off[n_hyp];
  if (n_out == 0) return PLLB_OK;
  e = cudaMemcpyAsync(d_ooff, out_off, 8 * (int64_t)(n_hyp + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) rc = launch_tokenize_write(d_table, table_size, d_cp, d_off, n_hyp, d_flag, d_ooff, d_ids, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(out_ids, d_ids, 4 * n_out, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaStreamSynchronize(s);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("pllb_tokenize_host: ") + cudaGetErrorString(e));
  return PLLB_OK;
}

int pllb_levenshtein_host(const int32_t* ref_cp, const int64_t* ref_off, int32_t n_ref, const int32_t* hyp_cp,
                          const int64_t* hyp_off, const int32_t* pair_ref, int32_t n_pairs, int32_t* out_dist) {
  RC(check_device());
  if (n_pairs <= 0) return PLLB_OK;
  if (!ref_off || !hyp_off || !pair_ref || !out_dist) return fail(PLLB_ERR_INVALID, "pllb_levenshtein_host: null argument");
  int32_t max_len = 0;
  for (int32_t i = 0; i < n_pairs; ++i) {
    max_len = std::max<int32_t>(max_len, (int32_t)(hyp_off[i + 1] - hyp_off[i]));
    if (pair_ref[i] < 0 || pair_ref[i] >= n_ref) return fail(PLLB_ERR_INVALID, "pllb_levenshtein_host: pair_ref out of range");
  }
  const int64_t n_rc = ref_off[n_ref], n_hc = hyp_off[n_pairs];
  const int64_t b0 = align_up(4 * std::max<int64_t>(n_rc, 1), 256), b1 = align_up(8 * (int64_t)(n_ref + 1), 256),
                b2 = align_up(4 * std::max<int64_t>(n_hc, 1), 256), b3 = align_up(8 * (int64_t)(n_pairs + 1), 256),
                b4 = align_up(4 * (int64_t)n_pairs, 256), b5 = b4;
  uint8_t* base = nullptr;
  RC(get_scratch(b0 + b1 + b2 + b3 + b4 + b5, &base));
  int32_t* d_rc = (int32_t*)base;
  int64_t* d_ro = (int64_t*)(base + b0);
  int32_t* d_hc = (int32_t*)(base + b0 + b1);
  int64_t* d_ho = (int64_t*)(base + b0 + b1 + b2);
  int32_t* d_pr = (int32_t*)(base + b0 + b1 + b2 + b3);
  int32_t* d_out = (int32_t*)(base + b0 + b1 + b2 + b3 + b4);
  cudaStream_t s = 0;
  int rc = PLLB_OK;
  cudaError_t e = cudaSuccess;
  if (n_rc > 0) e = cudaMemcpyAsync(d_rc, ref_cp, 4 * n_rc, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_ro, ref_off, 8 * (n_ref + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && n_hc > 0) e = cudaMemcpyAsync(d_hc, hyp_cp, 4 * n_hc, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_ho, hyp_off, 8 * (n_pairs + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_pr, pair_ref, 4 * (int64_t)n_pairs, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) rc = launch_levenshtein(d_rc, d_ro, d_hc, d_ho, d_pr, n_pairs, max_len, d_out, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(out_dist, d_out, 4 * (int64_t)n_pairs, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaStreamSynchronize(s);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("pllb_levenshtein_host: ") + cudaGetErrorString(e));
  return PLLB_OK;
}

int pllb_align(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
               const int32_t* pair_ref, int32_t n_pairs, int32_t max_len, const int64_t* ops_off, uint8_t* out_ops,
               int32_t* out_n_ops, int32_t* out_counts, void* stream) {
  RC(check_device());
  if (n_pairs <= 0) return PLLB_OK;
  if (max_len < 0) return fail(PLLB_ERR_INVALID, "pllb_align: negative max_len");
  if (max_len > 1024) return fail(PLLB_ERR_TOO_LONG, "pllb_align: max_len above 1024 symbols");
  NvtxRange r("stage4: align");
  int32_t warps = 0;
  int64_t slot_words = 0;
  align_shape(n_pairs, max_len, max_len, &warps, &slot_words);
  uint8_t* codes = nullptr;
  if (slot_words > 0) RC(get_scratch(8 * slot_words * warps, &codes));
  return launch_align(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref, n_pairs, max_len, max_len, ops_off, out_ops,
                      out_n_ops, out_counts, reinterpret_cast<uint2*>(codes), (cudaStream_t)stream);
}

int pllb_align_host(const int32_t* ref_cp, const int64_t* ref_off, int32_t n_ref, const int32_t* hyp_cp,
                    const int64_t* hyp_off, const int32_t* pair_ref, int32_t n_pairs, const int64_t* ops_off,
                    uint8_t* out_ops, int32_t* out_n_ops, int32_t* out_counts) {
  RC(check_device());
  if (n_pairs <= 0) return PLLB_OK;
  if (n_ref < 0 || !ref_off || !hyp_off || !pair_ref || !ops_off || !out_n_ops || !out_counts)
    return fail(PLLB_ERR_INVALID, "pllb_align_host: null argument");
  if (ref_off[0] < 0 || hyp_off[0] < 0 || ops_off[0] < 0) return fail(PLLB_ERR_INVALID, "pllb_align_host: negative offset");
  for (int32_t i = 0; i < n_ref; ++i)
    if (ref_off[i + 1] < ref_off[i]) return fail(PLLB_ERR_INVALID, "pllb_align_host: ref_off not ascending");
  int32_t max_ref = 0, max_hyp = 0;
  for (int32_t i = 0; i < n_pairs; ++i) {
    if (pair_ref[i] < 0 || pair_ref[i] >= n_ref) return fail(PLLB_ERR_INVALID, "pllb_align_host: pair_ref out of range");
    if (hyp_off[i + 1] < hyp_off[i]) return fail(PLLB_ERR_INVALID, "pllb_align_host: hyp_off not ascending");
    const int64_t na = ref_off[pair_ref[i] + 1] - ref_off[pair_ref[i]], nb = hyp_off[i + 1] - hyp_off[i];
    if (na > 1024 || nb > 1024) return fail(PLLB_ERR_TOO_LONG, "pllb_align_host: a side longer than 1024 symbols");
    if (ops_off[i + 1] - ops_off[i] < na + nb) return fail(PLLB_ERR_INVALID, "pllb_align_host: ops_off slot shorter than na + nb");
    max_ref = std::max<int32_t>(max_ref, (int32_t)na);
    max_hyp = std::max<int32_t>(max_hyp, (int32_t)nb);
  }
  const int64_t n_rc = ref_off[n_ref], n_hc = hyp_off[n_pairs], n_ops = ops_off[n_pairs];
  if ((n_rc > 0 && !ref_cp) || (n_hc > 0 && !hyp_cp) || (n_ops > 0 && !out_ops))
    return fail(PLLB_ERR_INVALID, "pllb_align_host: null argument");
  int32_t warps = 0;
  int64_t slot_words = 0;
  align_shape(n_pairs, max_ref, max_hyp, &warps, &slot_words);
  const int64_t b0 = align_up(4 * std::max<int64_t>(n_rc, 1), 256), b1 = align_up(8 * (int64_t)(n_ref + 1), 256),
                b2 = align_up(4 * std::max<int64_t>(n_hc, 1), 256), b3 = align_up(8 * (int64_t)(n_pairs + 1), 256),
                b4 = align_up(4 * (int64_t)n_pairs, 256), b5 = b3, b6 = align_up(std::max<int64_t>(n_ops, 1), 256),
                b7 = b4, b8 = align_up(16 * (int64_t)n_pairs, 256), b9 = 8 * slot_words * warps;
  uint8_t* base = nullptr;
  RC(get_scratch(b0 + b1 + b2 + b3 + b4 + b5 + b6 + b7 + b8 + b9, &base));
  int32_t* d_rc = (int32_t*)base;
  int64_t* d_ro = (int64_t*)(base + b0);
  int32_t* d_hc = (int32_t*)(base + b0 + b1);
  int64_t* d_ho = (int64_t*)(base + b0 + b1 + b2);
  int32_t* d_pr = (int32_t*)(base + b0 + b1 + b2 + b3);
  int64_t* d_oo = (int64_t*)(base + b0 + b1 + b2 + b3 + b4);
  uint8_t* d_ops = base + b0 + b1 + b2 + b3 + b4 + b5;
  int32_t* d_n = (int32_t*)(base + b0 + b1 + b2 + b3 + b4 + b5 + b6);
  int32_t* d_cnt = (int32_t*)(base + b0 + b1 + b2 + b3 + b4 + b5 + b6 + b7);
  uint2* d_codes = slot_words > 0 ? (uint2*)(base + b0 + b1 + b2 + b3 + b4 + b5 + b6 + b7 + b8) : nullptr;
  // ops are addressed relative to the first slot, so the device buffer starts at ops_off[0]
  std::vector<int64_t> rel(n_pairs + 1);
  for (int32_t i = 0; i <= n_pairs; ++i) rel[i] = ops_off[i] - ops_off[0];
  const int64_t n_out = rel[n_pairs];
  cudaStream_t s = 0;
  int rc = PLLB_OK;
  cudaError_t e = cudaSuccess;
  if (n_rc > 0) e = cudaMemcpyAsync(d_rc, ref_cp, 4 * n_rc, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_ro, ref_off, 8 * (int64_t)(n_ref + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && n_hc > 0) e = cudaMemcpyAsync(d_hc, hyp_cp, 4 * n_hc, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_ho, hyp_off, 8 * (int64_t)(n_pairs + 1), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_pr, pair_ref, 4 * (int64_t)n_pairs, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_oo, rel.data(), 8 * (int64_t)(n_pairs + 1), cudaMemcpyHostToDevice, s);
  // bytes of a slot past na + nb are not written by the kernel: zero them like its own padding
  if (e == cudaSuccess && n_out > 0) e = cudaMemsetAsync(d_ops, 0, n_out, s);
  if (e == cudaSuccess)
    rc = launch_align(d_rc, d_ro, d_hc, d_ho, d_pr, n_pairs, max_ref, max_hyp, d_oo, d_ops, d_n, d_cnt, d_codes, s);
  if (e == cudaSuccess && rc == PLLB_OK && n_out > 0)
    e = cudaMemcpyAsync(out_ops + ops_off[0], d_ops, n_out, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(out_n_ops, d_n, 4 * (int64_t)n_pairs, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(out_counts, d_cnt, 16 * (int64_t)n_pairs, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaStreamSynchronize(s);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("pllb_align_host: ") + cudaGetErrorString(e));
  return PLLB_OK;
}

int pllb_rescore_sweep(const double* am, const double* lm, const int64_t* len, const int32_t* dist, int32_t N,
                       int32_t n_best, const double* weights, int32_t W, int32_t variant, int32_t* out_argmax,
                       int64_t* out_edit_sum, void* stream) {
  RC(check_device());
  NvtxRange r("stage4: weight sweep");
  return launch_rescore_sweep(am, lm, len, dist, N, n_best, weights, W, variant, out_argmax, out_edit_sum,
                              (cudaStream_t)stream);
}

int pllb_rescore_sweep_host(const double* am, const double* lm, const int64_t* len, const int32_t* dist, int32_t N,
                            int32_t n_best, const double* weights, int32_t W, int32_t variant, int32_t* out_argmax,
                            int64_t* out_edit_sum) {
  RC(check_device());
  if (N <= 0 || W <= 0) return PLLB_OK;
  if (!am || !lm || !len || !weights || !out_argmax) return fail(PLLB_ERR_INVALID, "pllb_rescore_sweep_host: null argument");
  const int64_t n = (int64_t)N * n_best;
  const int64_t b_d = align_up(8 * n, 256), b_i = align_up(4 * n, 256), b_w = align_up(8 * (int64_t)W, 256),
                b_a = align_up(4 * (int64_t)W * N, 256);
  uint8_t* base = nullptr;
  RC(get_scratch(3 * b_d + b_i + 2 * b_w + b_a, &base));
  double* d_am = (double*)base;
  double* d_lm = (double*)(base + b_d);
  int64_t* d_len = (int64_t*)(base + 2 * b_d);
  int32_t* d_dist = (int32_t*)(base + 3 * b_d);
  double* d_w = (double*)(base + 3 * b_d + b_i);
  int64_t* d_es = (int64_t*)(base + 3 * b_d + b_i + b_w);
  int32_t* d_arg = (int32_t*)(base + 3 * b_d + b_i + 2 * b_w);
  cudaStream_t s = 0;
  int rc = PLLB_OK;
  cudaError_t e = cudaMemcpyAsync(d_am, am, 8 * n, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_lm, lm, 8 * n, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_len, len, 8 * n, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess && dist) e = cudaMemcpyAsync(d_dist, dist, 4 * n, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_w, weights, 8 * (int64_t)W, cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess)
    rc = launch_rescore_sweep(d_am, d_lm, d_len, dist ? d_dist : nullptr, N, n_best, d_w, W, variant, d_arg,
                              out_edit_sum ? d_es : nullptr, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaMemcpyAsync(out_argmax, d_arg, 4 * (int64_t)W * N, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK && out_edit_sum)
    e = cudaMemcpyAsync(out_edit_sum, d_es, 8 * (int64_t)W, cudaMemcpyDeviceToHost, s);
  if (e == cudaSuccess && rc == PLLB_OK) e = cudaStreamSynchronize(s);
  if (rc) return rc;
  if (e != cudaSuccess) return fail(PLLB_ERR_CUDA, std::string("pllb_rescore_sweep_host: ") + cudaGetErrorString(e));
  return PLLB_OK;
}

int pllb_rescore_scores(const double* am, const double* lm, const int64_t* len, int32_t N, int32_t n_best, double weight,
                        int32_t variant, double* out_scores, void* stream) {
  RC(check_device());
  return launch_rescore_scores(am, lm, len, N, n_best, weight, variant, out_scores, (cudaStream_t)stream);
}

}  // extern "C"
