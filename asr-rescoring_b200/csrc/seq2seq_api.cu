// seq2seq_api.cu — greedy encoder-decoder generation (include/pllb.h, pllb_s2s_* / pllb_generate*):
// CorrectBart's one_hyp correction.  The encoder is a pllb_handle driven through pllb_embed; the
// decoder step is the tcgen05 GEMM / GEMM+LayerNorm kernels with M = sentences in flight plus the
// small kernels of seq2seq_kernels.cu.  DESIGN.md §3.11.  Beam search (pllb_generate_beam*) runs the same
// decoder step over num_beams rows per sentence, with the EPI_TOPK head and beam_select_kernel.  §3.12.
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "common.h"

using namespace pllb;

namespace {

struct DecLayer {
  uint16_t *qkv_w, *o_w, *cq_w, *co_w, *ff1_w, *ff2_w;
  float *qkv_b, *o_b, *ln1_g, *ln1_b, *cq_b, *co_b, *ln2_g, *ln2_b, *ff1_b, *ff2_b, *ln3_g, *ln3_b;
};

#define RC(expr)            \
  do {                      \
    int _rc = (expr);       \
    if (_rc) return _rc;    \
  } while (0)

inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct pllb_s2s_ctx {
  pllb_s2s_desc d{};
  int device = 0;
  bool fp16 = false;
  int dt = DT_BF16;
  pllb_handle enc = nullptr;
  int32_t max_rows = 0;
  int64_t enc_cap = 0;                 // encoder rows of one chunk
  int vocab_pad = 0, tiles_v = 0;
  std::vector<void*> owned;
  int64_t owned_bytes = 0;
  // parameters
  float *word = nullptr;               // shared * embed_scale, fp32 (both embeddings)
  float *type_zero = nullptr, *dec_pos = nullptr, *dec_ln_g = nullptr, *dec_ln_b = nullptr;
  std::vector<DecLayer> layers;
  uint16_t* ckv_w = nullptr;           // [dec_layers * 2H, H]: layer l's K rows then V rows
  float* ckv_b = nullptr;
  uint16_t* head_w = nullptr;          // [vocab_pad, H], zero rows past vocab
  float* head_b = nullptr;             // final_logits_bias, zero past vocab
  // chunk workspace
  float *enc_f32 = nullptr, *hid32 = nullptr, *forced_logit = nullptr;
  uint16_t *enc16 = nullptr, *ckv = nullptr, *hid16 = nullptr, *wide = nullptr, *ctx = nullptr;
  float2* partials = nullptr;
  int32_t *force_col = nullptr, *done = nullptr, *enc_meta = nullptr;
  int32_t* meta_host = nullptr;        // pinned [2 * max_rows]
  int32_t* done_host = nullptr;        // pinned [2]
  cudaEvent_t ev_done[2] = {nullptr, nullptr};
  // KV cache, grown with max_length
  uint16_t* cache = nullptr;
  int64_t cache_elems = 0;
  // host-buffer entry point scratch
  void* io = nullptr;
  int64_t io_cap = 0;
  // beam search: per-row int32 / fp32 state and the EPI_TOPK partials, grown with max_length and KSEL
  void* beam = nullptr;
  int64_t beam_cap = 0;
  // stats / timing
  pllb_s2s_stats stats{};
  bool timing = false;
  std::vector<cudaEvent_t> evs;
};

namespace {

template <typename T>
int s2s_alloc(pllb_s2s_ctx* c, T** out, int64_t count) {
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

int copy_f32(pllb_s2s_ctx* c, float** dst, const float* src, int64_t n, cudaStream_t s) {
  if (!src) return fail(PLLB_ERR_INVALID, "pllb_s2s_create: null weight pointer");
  RC(s2s_alloc(c, dst, n));
  PLLB_CUDA(cudaMemcpyAsync(*dst, src, sizeof(float) * n, cudaMemcpyDeviceToDevice, s));
  return PLLB_OK;
}

// 16-bit copies of the row blocks srcs[i] ([rows_i, K] each) stacked in one [sum rows, K] operand
int conv_stack(pllb_s2s_ctx* c, uint16_t** dst, std::initializer_list<const float*> srcs, int64_t block, cudaStream_t s) {
  RC(s2s_alloc(c, dst, block * (int64_t)srcs.size()));
  int64_t i = 0;
  for (const float* p : srcs) {
    if (!p) return fail(PLLB_ERR_INVALID, "pllb_s2s_create: null weight pointer");
    RC(launch_f32_to_bf16(p, *dst + i * block, block, c->fp16, s));
    ++i;
  }
  return PLLB_OK;
}

int bias_stack(pllb_s2s_ctx* c, float** dst, std::initializer_list<const float*> srcs, int64_t block, cudaStream_t s) {
  RC(s2s_alloc(c, dst, block * (int64_t)srcs.size()));
  int64_t i = 0;
  for (const float* p : srcs) {
    if (!p) return fail(PLLB_ERR_INVALID, "pllb_s2s_create: null weight pointer");
    PLLB_CUDA(cudaMemcpyAsync(*dst + i * block, p, sizeof(float) * block, cudaMemcpyDeviceToDevice, s));
    ++i;
  }
  return PLLB_OK;
}

int check_s2s_desc(const pllb_s2s_desc& d) {
  const int H = d.hidden;
  if (H % 256 != 0 || H < 256 || H > 1024 || d.num_heads * 64 != H || d.enc_intermediate % 256 != 0 ||
      d.dec_intermediate % 256 != 0 || d.enc_intermediate < 256 || d.dec_intermediate < 256 || d.enc_layers < 1 ||
      d.dec_layers < 1 || d.vocab < 1 || d.enc_max_position < 3 || d.dec_max_position < 2 ||
      (d.operand_dtype != 0 && d.operand_dtype != 1) || !std::isfinite(d.embed_scale) || !(d.ln_eps > 0.f))
    return fail(PLLB_ERR_INVALID, "unsupported seq2seq shape: need hidden in {256,512,768,1024}, head dim 64, FFN "
                                  "widths % 256 == 0, >= 1 layer per stack, operand_dtype 0 or 1");
  if (d.cls_id < 0 || d.cls_id >= d.vocab || d.sep_id < 0 || d.sep_id >= d.vocab)
    return fail(PLLB_ERR_INVALID, "cls_id / sep_id outside the vocabulary");
  return PLLB_OK;
}

int check_gen_settings(const pllb_s2s_ctx* c, const pllb_gen_desc* g);

int check_gen(const pllb_s2s_ctx* c, const pllb_gen_desc* g) {
  if (!g) return fail(PLLB_ERR_INVALID, "pllb_generate: null generation settings");
  if (g->num_beams != 1)
    return fail(PLLB_ERR_INVALID, "pllb_generate is greedy (num_beams == 1); beam search is pllb_generate_beam");
  return check_gen_settings(c, g);
}

// every setting but num_beams, shared by greedy and beam search
int check_gen_settings(const pllb_s2s_ctx* c, const pllb_gen_desc* g) {
  if (g->do_sample != 0) return fail(PLLB_ERR_INVALID, "sampling is not supported");
  if (g->no_repeat_ngram_size != 0) return fail(PLLB_ERR_INVALID, "no_repeat_ngram_size is not supported");
  if (g->min_length != 0) return fail(PLLB_ERR_INVALID, "min_length is not supported");
  if (g->repetition_penalty != 1.0f) return fail(PLLB_ERR_INVALID, "repetition_penalty != 1 is not supported");
  if (g->max_length < 2 || g->max_length > c->d.dec_max_position)
    return fail(PLLB_ERR_INVALID, "max_length must lie in [2, " + std::to_string(c->d.dec_max_position) + "]");
  const int V = c->d.vocab;
  auto in_vocab = [V](int32_t id) { return id >= 0 && id < V; };
  if (!in_vocab(g->decoder_start_id) || !in_vocab(g->eos_id) || !in_vocab(g->pad_id))
    return fail(PLLB_ERR_INVALID, "decoder_start / eos / pad id outside the vocabulary");
  if ((g->forced_bos_id != -1 && !in_vocab(g->forced_bos_id)) || (g->forced_eos_id != -1 && !in_vocab(g->forced_eos_id)))
    return fail(PLLB_ERR_INVALID, "forced BOS / EOS id outside the vocabulary (-1 = none)");
  return PLLB_OK;
}

int check_beam(const pllb_s2s_ctx* c, const pllb_gen_desc* g, const pllb_beam_desc* bd) {
  if (!g || !bd) return fail(PLLB_ERR_INVALID, "pllb_generate_beam: null generation settings");
  const int K = g->num_beams;
  if (K < 2 || K > 8) return fail(PLLB_ERR_INVALID, "num_beams must lie in [2, 8]");
  if (c->d.vocab < 2 * K) return fail(PLLB_ERR_INVALID, "beam search needs vocab >= 2 * num_beams");
  if (c->max_rows < K) return fail(PLLB_ERR_INVALID, "max_rows < num_beams: a chunk must hold one sentence's beams");
  if (bd->num_return_sequences < 1 || bd->num_return_sequences > K)
    return fail(PLLB_ERR_INVALID, "num_return_sequences must lie in [1, num_beams]");
  if (!std::isfinite(bd->length_penalty)) return fail(PLLB_ERR_INVALID, "length_penalty must be finite");
  if (bd->early_stopping < 0 || bd->early_stopping > 2)
    return fail(PLLB_ERR_INVALID, "early_stopping must be 0 (False), 1 (True) or 2 (\"never\")");
  RC(check_gen_settings(c, g));
  if ((int64_t)K * g->max_length > 12288) return fail(PLLB_ERR_INVALID, "num_beams * max_length > 12288");
  return PLLB_OK;
}

int ensure_cache(pllb_s2s_ctx* c, int max_len) {
  const int64_t need = (int64_t)c->d.dec_layers * c->max_rows * max_len * 2 * c->d.hidden;
  if (need <= c->cache_elems) return PLLB_OK;
  PLLB_CUDA(cudaDeviceSynchronize());
  if (c->cache) {
    cudaFree(c->cache);
    c->owned_bytes -= c->cache_elems * 2;
    c->cache = nullptr;
    c->cache_elems = 0;
  }
  cudaError_t e = cudaMalloc(&c->cache, (size_t)need * 2);
  if (e != cudaSuccess) {
    cudaGetLastError();
    c->cache = nullptr;
    return fail(PLLB_ERR_OOM, "KV cache of " + std::to_string(need * 2) + " bytes does not fit; lower max_rows");
  }
  c->cache_elems = need;
  c->owned_bytes += need * 2;
  return PLLB_OK;
}

int record(pllb_s2s_ctx* c, size_t* used, cudaStream_t s) {
  if (!c->timing) return PLLB_OK;
  if (*used == c->evs.size()) {
    cudaEvent_t e;
    PLLB_CUDA(cudaEventCreate(&e));
    c->evs.push_back(e);
  }
  PLLB_CUDA(cudaEventRecord(c->evs[(*used)++], s));
  return PLLB_OK;
}

float elapsed(pllb_s2s_ctx* c, size_t a, size_t b) {
  float ms = 0.f;
  cudaEventElapsedTime(&ms, c->evs[a], c->evs[b]);
  return ms;
}

// One chunk of nb sentences (b .. b + nb) whose encoder rows total enc_rows.
int run_chunk(pllb_s2s_ctx* c, const pllb_gen_desc* g, const int32_t* tokens, const int64_t* off, int32_t b, int32_t nb,
              int64_t enc_rows, int max_T, int32_t* out_ids, int32_t* out_len, float* out_logit, cudaStream_t s) {
  const pllb_s2s_desc& d = c->d;
  const int H = d.hidden, NL = d.dec_layers, I = d.dec_intermediate, ML = g->max_length;
  const int dt = c->dt;
  size_t ev = 0;
  // encoder rows of every sentence: [CLS] t [SEP] packed back to back
  for (int32_t i = 0; i < nb; ++i) {
    c->meta_host[i] = (int32_t)(off[b + i] - off[b]) + 2 * i;
    c->meta_host[c->max_rows + i] = (int32_t)(off[b + i + 1] - off[b + i]) + 2;
  }
  PLLB_CUDA(cudaMemcpyAsync(c->enc_meta, c->meta_host, sizeof(int32_t) * 2 * c->max_rows, cudaMemcpyHostToDevice, s));
  const int32_t* enc_start = c->enc_meta;
  const int32_t* enc_len = c->enc_meta + c->max_rows;
  RC(record(c, &ev, s));                                                   // 0
  RC(pllb_embed(c->enc, tokens, off + b, nb, d.enc_layers, c->enc_f32, s));
  RC(launch_f32_to_bf16(c->enc_f32, c->enc16, enc_rows * H, c->fp16, s));
  RC(record(c, &ev, s));                                                   // 1
  // cross-attention K | V of every decoder layer in one GEMM over the encoder rows
  RC(launch_gemm_tcgen05(c->enc16, c->ckv_w, c->ckv_b, c->ckv, enc_rows, 2 * H * NL, H, EPI_BIAS_BF16, nullptr, dt, s));
  RC(record(c, &ev, s));                                                   // 2
  const double Hd = H, Ie = d.enc_intermediate, Id = I;
  c->stats.gemm_flops += (double)enc_rows * d.enc_layers * (8 * Hd * Hd + 4 * Hd * Ie) + (double)enc_rows * NL * 4 * Hd * Hd;

  DecodeState st{};
  st.ids = out_ids + (size_t)b * ML;
  st.logit = out_logit ? out_logit + (size_t)b * ML : nullptr;
  st.len = out_len + b;
  st.force_col = c->force_col;
  st.done_rows = c->done;
  st.rows = nb;
  st.max_len = ML;
  st.start_id = g->decoder_start_id;
  st.eos_id = g->eos_id;
  st.pad_id = g->pad_id;
  st.forced_bos = g->forced_bos_id;
  st.forced_eos = g->forced_eos_id;
  RC(launch_decode_init(st, s));
  const int64_t cache_layer = (int64_t)c->max_rows * ML * 2 * H;
  LseArgs head{c->force_col, c->partials, c->forced_logit, d.vocab};
  std::vector<size_t> step_ev;
  int64_t steps = 0;
  for (int t = 1; t < ML; ++t) {
    step_ev.push_back(ev);
    RC(record(c, &ev, s));
    RC(launch_dec_embed(st, t - 1, c->word, c->dec_pos, c->dec_ln_g, c->dec_ln_b, d.ln_eps, H, c->hid32, c->hid16, c->fp16, s));
    for (int l = 0; l < NL; ++l) {
      const DecLayer& L = c->layers[l];
      uint16_t* cache_l = c->cache + l * cache_layer;
      RC(launch_gemm_tcgen05(c->hid16, L.qkv_w, L.qkv_b, c->wide, nb, 3 * H, H, EPI_BIAS_BF16, nullptr, dt, s));
      RC(launch_decode_attention(c->wide, 3 * H, nullptr, 0, nullptr, nullptr, t - 1, ML, c->wide + H, 3 * H, cache_l,
                                 c->ctx, nb, H, ML, c->fp16, s));
      RC(launch_gemm_ln(c->ctx, L.o_w, L.o_b, L.ln1_g, L.ln1_b, d.ln_eps, c->hid32, c->hid16, nb, H, H, dt, s));
      RC(launch_gemm_tcgen05(c->hid16, L.cq_w, L.cq_b, c->wide, nb, H, H, EPI_BIAS_BF16, nullptr, dt, s));
      RC(launch_decode_attention(c->wide, H, c->ckv + (size_t)l * 2 * H, (int64_t)2 * H * NL, enc_start, enc_len, 0, ML,
                                 nullptr, 0, nullptr, c->ctx, nb, H, max_T, c->fp16, s));
      RC(launch_gemm_ln(c->ctx, L.co_w, L.co_b, L.ln2_g, L.ln2_b, d.ln_eps, c->hid32, c->hid16, nb, H, H, dt, s));
      RC(launch_gemm_tcgen05(c->hid16, L.ff1_w, L.ff1_b, c->wide, nb, I, H, EPI_BIAS_GELU_BF16, nullptr, dt, s));
      RC(launch_gemm_ln(c->wide, L.ff2_w, L.ff2_b, L.ln3_g, L.ln3_b, d.ln_eps, c->hid32, c->hid16, nb, H, I, dt, s));
    }
    RC(record(c, &ev, s));
    RC(launch_gemm_tcgen05(c->hid16, c->head_w, c->head_b, nullptr, nb, c->vocab_pad, H, EPI_ARGMAX, &head, dt, s));
    RC(launch_argmax_finish(c->partials, c->forced_logit, 2 * c->tiles_v, st, t, s));
    RC(record(c, &ev, s));
    ++steps;
    c->stats.gemm_flops += (double)nb * (NL * (12 * Hd * Hd + 4 * Hd * Id) + 2 * Hd * d.vocab);
    if (t == ML - 1) break;
    // finished-row count of this step; the host looks at the previous step's count, so the device
    // never idles waiting for the host.  A step run after every row finished writes pads over pads.
    PLLB_CUDA(cudaMemcpyAsync(c->done_host + (t & 1), c->done, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaEventRecord(c->ev_done[t & 1], s));
    if (t > 1) {
      PLLB_CUDA(cudaEventSynchronize(c->ev_done[(t - 1) & 1]));
      if (c->done_host[(t - 1) & 1] >= nb) break;
    }
  }
  PLLB_CUDA(cudaStreamSynchronize(s));
  c->stats.steps += steps;
  if (c->timing) {
    c->stats.enc_ms += elapsed(c, 0, 1);
    c->stats.cross_kv_ms += elapsed(c, 1, 2);
    for (size_t e : step_ev) {
      c->stats.dec_layers_ms += elapsed(c, e, e + 1);
      c->stats.head_ms += elapsed(c, e + 1, e + 2);
    }
    c->stats.total_ms += elapsed(c, 0, ev - 1);
  }
  return PLLB_OK;
}

int generate_impl(pllb_s2s_ctx* c, const pllb_gen_desc* g, const int32_t* tokens, const int64_t* off, int32_t n,
                  int32_t* out_ids, int32_t* out_len, float* out_logit, cudaStream_t s) {
  if (!c) return fail(PLLB_ERR_INVALID, "null handle");
  RC(check_gen(c, g));
  if (n < 0) return fail(PLLB_ERR_INVALID, "pllb_generate: negative sentence count");
  if (n == 0) return PLLB_OK;
  if (!off || !out_ids || !out_len) return fail(PLLB_ERR_INVALID, "pllb_generate: null argument");
  if (!tokens && off[n] > off[0]) return fail(PLLB_ERR_INVALID, "pllb_generate: tokens is null");
  for (int32_t i = 0; i < n; ++i) {
    const int64_t L = off[i + 1] - off[i];
    if (L < 0) return fail(PLLB_ERR_INVALID, "pllb_generate: offsets not monotone");
    if (L + 2 > c->d.enc_max_position)
      return fail(PLLB_ERR_TOO_LONG, "sentence " + std::to_string(i) + " has " + std::to_string(L) +
                                         " tokens; max_position_embeddings allows " + std::to_string(c->d.enc_max_position - 2));
  }
  PLLB_CUDA(cudaSetDevice(c->device));
  RC(ensure_cache(c, g->max_length));
  const int64_t launches_before = g_launch_counter;
  if (c->timing) c->stats.enc_ms = c->stats.cross_kv_ms = c->stats.dec_layers_ms = c->stats.head_ms = c->stats.total_ms = 0.f;
  int32_t b = 0;
  while (b < n) {
    int32_t e = b;
    int64_t rows = 0;
    int max_T = 0;
    while (e < n && e - b < c->max_rows) {
      const int64_t T = off[e + 1] - off[e] + 2;
      if (e > b && rows + T > c->enc_cap) break;
      rows += T;
      max_T = std::max<int>(max_T, (int)T);
      ++e;
    }
    RC(run_chunk(c, g, tokens, off, b, e - b, rows, max_T, out_ids, out_len, out_logit, s));
    c->stats.chunks += 1;
    c->stats.sentences += e - b;
    b = e;
  }
  c->stats.kernel_launches += g_launch_counter - launches_before;
  return PLLB_OK;
}


// ------------------------------------------------------------------------------------ beam search
int ksel_of(int K) { return K <= 4 ? 8 : 16; }

// Carves the beam state of a chunk of max_rows / K sentences out of one growing allocation.
int beam_state(pllb_s2s_ctx* c, const pllb_gen_desc* g, const pllb_beam_desc* bd, int32_t nb, BeamState* st,
               float2** topk) {
  const int K = g->num_beams, ML = g->max_length;
  const int64_t R = c->max_rows;
  const int64_t parts = R * 2 * c->tiles_v * (1 + ksel_of(K));
  const int64_t b_i32 = align_up(sizeof(int32_t) * (R * ML * 5 + R * 3 + R + 1), 256);
  const int64_t b_f32 = align_up(sizeof(float) * R * 2, 256);
  const int64_t need = b_i32 + b_f32 + (int64_t)sizeof(float2) * parts;
  if (need > c->beam_cap) {
    PLLB_CUDA(cudaDeviceSynchronize());
    if (c->beam) cudaFree(c->beam);
    c->owned_bytes -= c->beam_cap;
    c->beam = nullptr;
    c->beam_cap = 0;
    cudaError_t e = cudaMalloc(&c->beam, (size_t)need);
    if (e != cudaSuccess) {
      cudaGetLastError();
      c->beam = nullptr;
      return fail(PLLB_ERR_OOM, "beam search state of " + std::to_string(need) + " bytes does not fit; lower max_rows");
    }
    c->beam_cap = need;
    c->owned_bytes += need;
  }
  int32_t* p = reinterpret_cast<int32_t*>(c->beam);
  const int64_t RL = R * ML;
  BeamState b{};
  int32_t* ids0 = p;
  int32_t* ids1 = p + RL;
  b.ids_cur = ids0;
  b.ids_next = ids1;
  b.slot_cur = p + 2 * RL;
  b.slot_next = p + 3 * RL;
  b.fin_ids = p + 4 * RL;
  b.parent = p + 5 * RL;
  b.fin_len = p + 5 * RL + R;
  b.fin_flag = p + 5 * RL + 2 * R;
  b.sent_flags = p + 5 * RL + 3 * R;
  b.frozen_count = p + 5 * RL + 4 * R;
  float* f = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(c->beam) + b_i32);
  b.run_score = f;
  b.fin_score = f + R;
  *topk = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(c->beam) + b_i32 + b_f32);
  b.n = nb;
  b.K = K;
  b.max_len = ML;
  b.start_id = g->decoder_start_id;
  b.eos_id = g->eos_id;
  b.pad_id = g->pad_id;
  b.forced_bos = g->forced_bos_id;
  b.forced_eos = g->forced_eos_id;
  b.early_stopping = bd->early_stopping;
  b.length_penalty = bd->length_penalty;
  *st = b;
  return PLLB_OK;
}

// The head of step t over hid16 (n * K rows): EPI_TOPK GEMM, beam_select_kernel, then the ping-pong swap.
int beam_head_step(pllb_s2s_ctx* c, BeamState* st, float2* topk, int t, cudaStream_t s) {
  const int K = st->K, ksel = ksel_of(K);
  const int64_t R = (int64_t)st->n * K;
  LseArgs head{nullptr, topk, nullptr, c->d.vocab};
  RC(launch_gemm_tcgen05(c->hid16, c->head_w, c->head_b, nullptr, R, c->vocab_pad, c->d.hidden,
                         ksel == 8 ? EPI_TOPK8 : EPI_TOPK16, &head, c->dt, s));
  RC(launch_beam_select(topk, 2 * c->tiles_v, ksel, c->d.vocab, *st, t, s));
  std::swap(st->ids_cur, st->ids_next);
  std::swap(st->slot_cur, st->slot_next);
  return PLLB_OK;
}

// One chunk of nb sentences (b .. b + nb), nb * K decoder rows.
int run_chunk_beam(pllb_s2s_ctx* c, const pllb_gen_desc* g, const pllb_beam_desc* bd, const int32_t* tokens,
                   const int64_t* off, int32_t b, int32_t nb, int64_t enc_rows, int max_T, int32_t* out_ids,
                   int32_t* out_len, float* out_score, cudaStream_t s) {
  const pllb_s2s_desc& d = c->d;
  const int H = d.hidden, NL = d.dec_layers, I = d.dec_intermediate, ML = g->max_length, K = g->num_beams;
  const int R = nb * K, dt = c->dt, nr = bd->num_return_sequences;
  size_t ev = 0;
  // every beam row reads its sentence's encoder rows
  for (int32_t i = 0; i < nb; ++i)
    for (int k = 0; k < K; ++k) {
      c->meta_host[i * K + k] = (int32_t)(off[b + i] - off[b]) + 2 * i;
      c->meta_host[c->max_rows + i * K + k] = (int32_t)(off[b + i + 1] - off[b + i]) + 2;
    }
  PLLB_CUDA(cudaMemcpyAsync(c->enc_meta, c->meta_host, sizeof(int32_t) * 2 * c->max_rows, cudaMemcpyHostToDevice, s));
  const int32_t* enc_start = c->enc_meta;
  const int32_t* enc_len = c->enc_meta + c->max_rows;
  RC(record(c, &ev, s));                                                   // 0
  RC(pllb_embed(c->enc, tokens, off + b, nb, d.enc_layers, c->enc_f32, s));
  RC(launch_f32_to_bf16(c->enc_f32, c->enc16, enc_rows * H, c->fp16, s));
  RC(record(c, &ev, s));                                                   // 1
  RC(launch_gemm_tcgen05(c->enc16, c->ckv_w, c->ckv_b, c->ckv, enc_rows, 2 * H * NL, H, EPI_BIAS_BF16, nullptr, dt, s));
  RC(record(c, &ev, s));                                                   // 2
  const double Hd = H, Ie = d.enc_intermediate, Id = I;
  c->stats.gemm_flops += (double)enc_rows * d.enc_layers * (8 * Hd * Hd + 4 * Hd * Ie) + (double)enc_rows * NL * 4 * Hd * Hd;

  BeamState st{};
  float2* topk = nullptr;
  RC(beam_state(c, g, bd, nb, &st, &topk));
  RC(launch_beam_init(st, s));
  DecodeState ds{};
  ds.rows = R;
  ds.max_len = ML;
  const int64_t cache_layer = (int64_t)c->max_rows * ML * 2 * H;
  std::vector<size_t> step_ev;
  int64_t steps = 0;
  for (int t = 1; t < ML; ++t) {
    step_ev.push_back(ev);
    RC(record(c, &ev, s));
    ds.ids = st.ids_cur;
    RC(launch_dec_embed(ds, t - 1, c->word, c->dec_pos, c->dec_ln_g, c->dec_ln_b, d.ln_eps, H, c->hid32, c->hid16, c->fp16, s));
    for (int l = 0; l < NL; ++l) {
      const DecLayer& L = c->layers[l];
      uint16_t* cache_l = c->cache + l * cache_layer;
      RC(launch_gemm_tcgen05(c->hid16, L.qkv_w, L.qkv_b, c->wide, R, 3 * H, H, EPI_BIAS_BF16, nullptr, dt, s));
      RC(launch_decode_attention(c->wide, 3 * H, nullptr, 0, nullptr, nullptr, t - 1, ML, c->wide + H, 3 * H, cache_l,
                                 c->ctx, R, H, ML, c->fp16, s, st.slot_cur));
      RC(launch_gemm_ln(c->ctx, L.o_w, L.o_b, L.ln1_g, L.ln1_b, d.ln_eps, c->hid32, c->hid16, R, H, H, dt, s));
      RC(launch_gemm_tcgen05(c->hid16, L.cq_w, L.cq_b, c->wide, R, H, H, EPI_BIAS_BF16, nullptr, dt, s));
      RC(launch_decode_attention(c->wide, H, c->ckv + (size_t)l * 2 * H, (int64_t)2 * H * NL, enc_start, enc_len, 0, ML,
                                 nullptr, 0, nullptr, c->ctx, R, H, max_T, c->fp16, s));
      RC(launch_gemm_ln(c->ctx, L.co_w, L.co_b, L.ln2_g, L.ln2_b, d.ln_eps, c->hid32, c->hid16, R, H, H, dt, s));
      RC(launch_gemm_tcgen05(c->hid16, L.ff1_w, L.ff1_b, c->wide, R, I, H, EPI_BIAS_GELU_BF16, nullptr, dt, s));
      RC(launch_gemm_ln(c->wide, L.ff2_w, L.ff2_b, L.ln3_g, L.ln3_b, d.ln_eps, c->hid32, c->hid16, R, H, I, dt, s));
    }
    RC(record(c, &ev, s));
    RC(beam_head_step(c, &st, topk, t, s));                               // head GEMM + selection: head_ms
    RC(record(c, &ev, s));
    ++steps;
    c->stats.gemm_flops += (double)R * (NL * (12 * Hd * Hd + 4 * Hd * Id) + 2 * Hd * d.vocab);
    if (t == ML - 1) break;
    // frozen-sentence count, read one step late as greedy reads its finished-row count
    PLLB_CUDA(cudaMemcpyAsync(c->done_host + (t & 1), st.frozen_count, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaEventRecord(c->ev_done[t & 1], s));
    if (t > 1) {
      PLLB_CUDA(cudaEventSynchronize(c->ev_done[(t - 1) & 1]));
      if (c->done_host[(t - 1) & 1] >= nb) break;
    }
  }
  RC(launch_beam_output(st, nr, out_ids + (size_t)b * nr * ML, out_len + (size_t)b * nr, out_score + (size_t)b * nr, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  c->stats.steps += steps;
  if (c->timing) {
    c->stats.enc_ms += elapsed(c, 0, 1);
    c->stats.cross_kv_ms += elapsed(c, 1, 2);
    for (size_t e : step_ev) {
      c->stats.dec_layers_ms += elapsed(c, e, e + 1);
      c->stats.head_ms += elapsed(c, e + 1, e + 2);
    }
    c->stats.total_ms += elapsed(c, 0, ev - 1);
  }
  return PLLB_OK;
}

int check_inputs(const pllb_s2s_ctx* c, const int32_t* tokens, const int64_t* off, int32_t n, const void* a,
                 const void* b, const void* d, const char* who) {
  if (n < 0) return fail(PLLB_ERR_INVALID, std::string(who) + ": negative sentence count");
  if (n == 0) return PLLB_OK;
  if (!off || !a || !b || !d) return fail(PLLB_ERR_INVALID, std::string(who) + ": null argument");
  if (!tokens && off[n] > off[0]) return fail(PLLB_ERR_INVALID, std::string(who) + ": tokens is null");
  for (int32_t i = 0; i < n; ++i) {
    const int64_t L = off[i + 1] - off[i];
    if (L < 0) return fail(PLLB_ERR_INVALID, std::string(who) + ": offsets not monotone");
    if (L + 2 > c->d.enc_max_position)
      return fail(PLLB_ERR_TOO_LONG, "sentence " + std::to_string(i) + " has " + std::to_string(L) +
                                         " tokens; max_position_embeddings allows " + std::to_string(c->d.enc_max_position - 2));
  }
  return PLLB_OK;
}

int generate_beam_impl(pllb_s2s_ctx* c, const pllb_gen_desc* g, const pllb_beam_desc* bd, const int32_t* tokens,
                       const int64_t* off, int32_t n, int32_t* out_ids, int32_t* out_len, float* out_score,
                       cudaStream_t s) {
  if (!c) return fail(PLLB_ERR_INVALID, "null handle");
  RC(check_beam(c, g, bd));
  RC(check_inputs(c, tokens, off, n, out_ids, out_len, out_score, "pllb_generate_beam"));
  if (n == 0) return PLLB_OK;
  PLLB_CUDA(cudaSetDevice(c->device));
  RC(ensure_cache(c, g->max_length));
  const int K = g->num_beams;
  const int32_t per_chunk = c->max_rows / K;
  const int64_t launches_before = g_launch_counter;
  if (c->timing) c->stats.enc_ms = c->stats.cross_kv_ms = c->stats.dec_layers_ms = c->stats.head_ms = c->stats.total_ms = 0.f;
  int32_t b = 0;
  while (b < n) {
    int32_t e = b;
    int64_t rows = 0;
    int max_T = 0;
    while (e < n && e - b < per_chunk) {
      const int64_t T = off[e + 1] - off[e] + 2;
      if (e > b && rows + T > c->enc_cap) break;
      rows += T;
      max_T = std::max<int>(max_T, (int)T);
      ++e;
    }
    RC(run_chunk_beam(c, g, bd, tokens, off, b, e - b, rows, max_T, out_ids, out_len, out_score, s));
    c->stats.chunks += 1;
    c->stats.sentences += e - b;
    b = e;
  }
  c->stats.kernel_launches += g_launch_counter - launches_before;
  return PLLB_OK;
}

}  // namespace

extern "C" {

int pllb_s2s_create(pllb_s2s* out, const pllb_s2s_desc* desc, const pllb_s2s_weights* w, int32_t max_rows, int device) {
  if (!out || !desc || !w || !w->enc.layers || !w->dec_layers || !w->shared)
    return fail(PLLB_ERR_INVALID, "pllb_s2s_create: null argument");
  *out = nullptr;
  const pllb_s2s_desc& d = *desc;
  RC(check_s2s_desc(d));
  if (max_rows < 0) return fail(PLLB_ERR_INVALID, "pllb_s2s_create: max_rows < 0");
  if (pllb_device_count() < 1) return fail(PLLB_ERR_NO_DEVICE, "no sm_100 device visible; libpllb200 has no CPU fallback");
  PLLB_CUDA(cudaSetDevice(device));
  int major = 0;
  PLLB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(PLLB_ERR_NO_DEVICE, "device is not sm_100 (B200); libpllb200 has no other code path");
  pllb_s2s_ctx* c = new pllb_s2s_ctx();
  c->d = d;
  c->device = device;
  c->fp16 = d.operand_dtype == 1;
  c->dt = c->fp16 ? DT_FP16 : DT_BF16;
  c->max_rows = max_rows > 0 ? max_rows : 8192;
  c->enc_cap = std::max<int64_t>((int64_t)c->max_rows * 32, d.enc_max_position);
  const int H = d.hidden, V = d.vocab, NL = d.dec_layers, I = d.dec_intermediate;
  c->vocab_pad = (int)align_up(V, 256);
  c->tiles_v = c->vocab_pad / 256;
  cudaStream_t s = 0;
  int rc = PLLB_OK;
#define TRY(expr)                            \
  do {                                       \
    rc = (expr);                             \
    if (rc) { pllb_s2s_destroy(c); return rc; } \
  } while (0)
  // token table * embed_scale: the lookups of both embeddings (never the LM head)
  TRY(s2s_alloc(c, &c->word, (int64_t)V * H));
  TRY(launch_scale_copy(w->shared, c->word, (int64_t)V * H, d.embed_scale, s));
  TRY(s2s_alloc(c, &c->type_zero, H));
  if (cudaMemsetAsync(c->type_zero, 0, sizeof(float) * H, s) != cudaSuccess) TRY(fail(PLLB_ERR_CUDA, "memset"));
  {
    pllb_model_desc ed{};
    ed.num_layers = d.enc_layers;
    ed.hidden = H;
    ed.num_heads = d.num_heads;
    ed.intermediate = d.enc_intermediate;
    ed.vocab = V;
    ed.max_position = d.enc_max_position;
    ed.ln_eps = d.ln_eps;
    ed.cls_id = d.cls_id;
    ed.sep_id = d.sep_id;
    ed.mask_id = d.cls_id;       // no masked copies on this path
    ed.operand_dtype = d.operand_dtype;
    pllb_weights ew = w->enc;
    ew.word_emb = c->word;
    ew.type_emb = c->type_zero;
    ew.head_w = ew.head_b = ew.head_ln_g = ew.head_ln_b = ew.decoder_w = ew.decoder_b = nullptr;
    if (cudaStreamSynchronize(s) != cudaSuccess) TRY(fail(PLLB_ERR_CUDA, "pllb_s2s_create: weight copy failed"));
    TRY(pllb_create(&c->enc, &ed, &ew, c->enc_cap, device));
  }
  TRY(copy_f32(c, &c->dec_pos, w->dec_pos_emb, (int64_t)d.dec_max_position * H, s));
  TRY(copy_f32(c, &c->dec_ln_g, w->dec_emb_ln_g, H, s));
  TRY(copy_f32(c, &c->dec_ln_b, w->dec_emb_ln_b, H, s));
  c->layers.resize(NL);
  const int64_t HH = (int64_t)H * H;
  std::vector<const float*> ckw, ckb;
  for (int l = 0; l < NL; ++l) {
    const pllb_dec_layer_weights& lw = w->dec_layers[l];
    DecLayer& L = c->layers[l];
    TRY(conv_stack(c, &L.qkv_w, {lw.q_w, lw.k_w, lw.v_w}, HH, s));
    TRY(bias_stack(c, &L.qkv_b, {lw.q_b, lw.k_b, lw.v_b}, H, s));
    TRY(conv_stack(c, &L.o_w, {lw.o_w}, HH, s));
    TRY(copy_f32(c, &L.o_b, lw.o_b, H, s));
    TRY(copy_f32(c, &L.ln1_g, lw.self_ln_g, H, s));
    TRY(copy_f32(c, &L.ln1_b, lw.self_ln_b, H, s));
    TRY(conv_stack(c, &L.cq_w, {lw.cq_w}, HH, s));
    TRY(copy_f32(c, &L.cq_b, lw.cq_b, H, s));
    TRY(conv_stack(c, &L.co_w, {lw.co_w}, HH, s));
    TRY(copy_f32(c, &L.co_b, lw.co_b, H, s));
    TRY(copy_f32(c, &L.ln2_g, lw.cross_ln_g, H, s));
    TRY(copy_f32(c, &L.ln2_b, lw.cross_ln_b, H, s));
    TRY(conv_stack(c, &L.ff1_w, {lw.ff1_w}, (int64_t)I * H, s));
    TRY(copy_f32(c, &L.ff1_b, lw.ff1_b, I, s));
    TRY(conv_stack(c, &L.ff2_w, {lw.ff2_w}, (int64_t)H * I, s));
    TRY(copy_f32(c, &L.ff2_b, lw.ff2_b, H, s));
    TRY(copy_f32(c, &L.ln3_g, lw.final_ln_g, H, s));
    TRY(copy_f32(c, &L.ln3_b, lw.final_ln_b, H, s));
  }
  TRY(s2s_alloc(c, &c->ckv_w, (int64_t)NL * 2 * HH));
  TRY(s2s_alloc(c, &c->ckv_b, (int64_t)NL * 2 * H));
  for (int l = 0; l < NL; ++l) {
    const pllb_dec_layer_weights& lw = w->dec_layers[l];
    if (!lw.ck_w || !lw.cv_w || !lw.ck_b || !lw.cv_b) TRY(fail(PLLB_ERR_INVALID, "pllb_s2s_create: null weight pointer"));
    TRY(launch_f32_to_bf16(lw.ck_w, c->ckv_w + (int64_t)l * 2 * HH, HH, c->fp16, s));
    TRY(launch_f32_to_bf16(lw.cv_w, c->ckv_w + (int64_t)l * 2 * HH + HH, HH, c->fp16, s));
    if (cudaMemcpyAsync(c->ckv_b + (int64_t)l * 2 * H, lw.ck_b, sizeof(float) * H, cudaMemcpyDeviceToDevice, s) ||
        cudaMemcpyAsync(c->ckv_b + (int64_t)l * 2 * H + H, lw.cv_b, sizeof(float) * H, cudaMemcpyDeviceToDevice, s))
      TRY(fail(PLLB_ERR_CUDA, "pllb_s2s_create: bias copy failed"));
  }
  if (!w->final_logits_bias) TRY(fail(PLLB_ERR_INVALID, "pllb_s2s_create: final_logits_bias is null"));
  TRY(s2s_alloc(c, &c->head_w, (int64_t)c->vocab_pad * H));
  TRY(s2s_alloc(c, &c->head_b, c->vocab_pad));
  if (cudaMemsetAsync(c->head_w, 0, sizeof(uint16_t) * (size_t)c->vocab_pad * H, s) ||
      cudaMemsetAsync(c->head_b, 0, sizeof(float) * c->vocab_pad, s) ||
      cudaMemcpyAsync(c->head_b, w->final_logits_bias, sizeof(float) * V, cudaMemcpyDeviceToDevice, s))
    TRY(fail(PLLB_ERR_CUDA, "pllb_s2s_create: head copy failed"));
  TRY(launch_f32_to_bf16(w->shared, c->head_w, (int64_t)V * H, c->fp16, s));
  // chunk workspace
  const int64_t R = c->max_rows, E = c->enc_cap;
  TRY(s2s_alloc(c, &c->enc_f32, E * H));
  TRY(s2s_alloc(c, &c->enc16, E * H));
  TRY(s2s_alloc(c, &c->ckv, E * 2 * H * NL));
  TRY(s2s_alloc(c, &c->hid32, align_up(R, 256) * H));     // T32 layout, padded to the LayerNorm clusters' blocks
  TRY(s2s_alloc(c, &c->hid16, R * H));
  TRY(s2s_alloc(c, &c->wide, R * std::max(3 * H, I)));
  TRY(s2s_alloc(c, &c->ctx, R * H));
  TRY(s2s_alloc(c, &c->partials, R * 2 * c->tiles_v));
  TRY(s2s_alloc(c, &c->forced_logit, R));
  TRY(s2s_alloc(c, &c->force_col, R));
  TRY(s2s_alloc(c, &c->done, 1));
  TRY(s2s_alloc(c, &c->enc_meta, 2 * R));
  if (cudaHostAlloc(&c->meta_host, sizeof(int32_t) * 2 * R, cudaHostAllocDefault) != cudaSuccess ||
      cudaHostAlloc(&c->done_host, sizeof(int32_t) * 2, cudaHostAllocDefault) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_done[0], cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_done[1], cudaEventDisableTiming) != cudaSuccess)
    TRY(fail(PLLB_ERR_CUDA, "pllb_s2s_create: pinned buffers / events"));
#undef TRY
  cudaError_t e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) {
    pllb_s2s_destroy(c);
    return fail(PLLB_ERR_CUDA, std::string("pllb_s2s_create: ") + cudaGetErrorString(e));
  }
  *out = c;
  return PLLB_OK;
}

int pllb_s2s_destroy(pllb_s2s h) {
  if (!h) return PLLB_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  if (h->enc) pllb_destroy(h->enc);
  for (void* p : h->owned) cudaFree(p);
  if (h->cache) cudaFree(h->cache);
  if (h->io) cudaFree(h->io);
  if (h->beam) cudaFree(h->beam);
  if (h->meta_host) cudaFreeHost(h->meta_host);
  if (h->done_host) cudaFreeHost(h->done_host);
  for (cudaEvent_t e : h->ev_done)
    if (e) cudaEventDestroy(e);
  for (cudaEvent_t e : h->evs) cudaEventDestroy(e);
  delete h;
  return PLLB_OK;
}

int64_t pllb_s2s_workspace_bytes(pllb_s2s h) {
  return h ? h->owned_bytes + pllb_workspace_bytes(h->enc) : 0;
}

int pllb_s2s_set_timing(pllb_s2s h, int enable) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  h->timing = enable != 0;
  return PLLB_OK;
}

int pllb_s2s_get_stats(pllb_s2s h, pllb_s2s_stats* out) {
  if (!h || !out) return fail(PLLB_ERR_INVALID, "pllb_s2s_get_stats: null argument");
  *out = h->stats;
  return PLLB_OK;
}

int pllb_s2s_reset_stats(pllb_s2s h) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  h->stats = pllb_s2s_stats{};
  return PLLB_OK;
}

int pllb_generate(pllb_s2s h, const pllb_gen_desc* gen, const int32_t* tokens, const int64_t* offsets, int32_t n,
                  int32_t* out_ids, int32_t* out_len, float* out_logit, void* stream) {
  return generate_impl(h, gen, tokens, offsets, n, out_ids, out_len, out_logit, (cudaStream_t)stream);
}

int pllb_generate_host(pllb_s2s h, const pllb_gen_desc* gen, const int32_t* tokens, const int64_t* off, int32_t n,
                       int32_t* out_ids, int32_t* out_len, float* out_logit) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  RC(check_gen(h, gen));
  if (n < 0) return fail(PLLB_ERR_INVALID, "pllb_generate_host: negative sentence count");
  if (n == 0) return PLLB_OK;
  if (!off || !out_ids || !out_len) return fail(PLLB_ERR_INVALID, "pllb_generate_host: null argument");
  const int64_t n_tok = off[n] - off[0];
  if (n_tok < 0) return fail(PLLB_ERR_INVALID, "pllb_generate_host: offsets not monotone");
  if (n_tok > 0 && !tokens) return fail(PLLB_ERR_INVALID, "pllb_generate_host: tokens is null");
  // the reference's embedding lookup raises IndexError on an id outside the vocabulary
  for (int64_t i = off[0]; i < off[n]; ++i)
    if (tokens[i] < 0 || tokens[i] >= h->d.vocab)
      return fail(PLLB_ERR_INVALID, "token id " + std::to_string(tokens[i]) + " at position " + std::to_string(i) +
                                        " is outside the vocabulary [0, " + std::to_string(h->d.vocab) + ")");
  PLLB_CUDA(cudaSetDevice(h->device));
  const int64_t ML = gen->max_length;
  const int64_t b_tok = align_up(sizeof(int32_t) * std::max<int64_t>(n_tok, 1), 256);
  const int64_t b_ids = align_up(sizeof(int32_t) * n * ML, 256);
  const int64_t b_len = align_up(sizeof(int32_t) * n, 256);
  const int64_t b_lg = out_logit ? align_up(sizeof(float) * n * ML, 256) : 0;
  const int64_t need = b_tok + b_ids + b_len + b_lg;
  if (need > h->io_cap) {
    PLLB_CUDA(cudaDeviceSynchronize());
    if (h->io) cudaFree(h->io);
    h->io = nullptr;
    h->io_cap = 0;
    PLLB_CUDA(cudaMalloc(&h->io, (size_t)need));
    h->io_cap = need;
  }
  uint8_t* base = reinterpret_cast<uint8_t*>(h->io);
  int32_t* d_tok = reinterpret_cast<int32_t*>(base);
  int32_t* d_ids = reinterpret_cast<int32_t*>(base + b_tok);
  int32_t* d_len = reinterpret_cast<int32_t*>(base + b_tok + b_ids);
  float* d_lg = out_logit ? reinterpret_cast<float*>(base + b_tok + b_ids + b_len) : nullptr;
  cudaStream_t s = 0;
  if (n_tok > 0) PLLB_CUDA(cudaMemcpyAsync(d_tok, tokens + off[0], sizeof(int32_t) * n_tok, cudaMemcpyHostToDevice, s));
  // the device tokens start at off[0]: index them from there
  RC(generate_impl(h, gen, d_tok - off[0], off, n, d_ids, d_len, d_lg, s));
  PLLB_CUDA(cudaMemcpyAsync(out_ids, d_ids, sizeof(int32_t) * n * ML, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaMemcpyAsync(out_len, d_len, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, s));
  if (out_logit) PLLB_CUDA(cudaMemcpyAsync(out_logit, d_lg, sizeof(float) * n * ML, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  return PLLB_OK;
}

int pllb_generate_beam(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, const int32_t* tokens,
                       const int64_t* offsets, int32_t n, int32_t* out_ids, int32_t* out_len, float* out_score,
                       void* stream) {
  return generate_beam_impl(h, gen, beam, tokens, offsets, n, out_ids, out_len, out_score, (cudaStream_t)stream);
}

int pllb_generate_beam_host(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, const int32_t* tokens,
                            const int64_t* off, int32_t n, int32_t* out_ids, int32_t* out_len, float* out_score) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  RC(check_beam(h, gen, beam));
  if (n < 0) return fail(PLLB_ERR_INVALID, "pllb_generate_beam_host: negative sentence count");
  if (n == 0) return PLLB_OK;
  if (!off || !out_ids || !out_len || !out_score) return fail(PLLB_ERR_INVALID, "pllb_generate_beam_host: null argument");
  const int64_t n_tok = off[n] - off[0];
  if (n_tok < 0) return fail(PLLB_ERR_INVALID, "pllb_generate_beam_host: offsets not monotone");
  if (n_tok > 0 && !tokens) return fail(PLLB_ERR_INVALID, "pllb_generate_beam_host: tokens is null");
  for (int64_t i = off[0]; i < off[n]; ++i)
    if (tokens[i] < 0 || tokens[i] >= h->d.vocab)
      return fail(PLLB_ERR_INVALID, "token id " + std::to_string(tokens[i]) + " at position " + std::to_string(i) +
                                        " is outside the vocabulary [0, " + std::to_string(h->d.vocab) + ")");
  PLLB_CUDA(cudaSetDevice(h->device));
  const int64_t ML = gen->max_length, nr = beam->num_return_sequences;
  const int64_t b_tok = align_up(sizeof(int32_t) * std::max<int64_t>(n_tok, 1), 256);
  const int64_t b_ids = align_up(sizeof(int32_t) * n * nr * ML, 256);
  const int64_t b_len = align_up(sizeof(int32_t) * n * nr, 256);
  const int64_t b_sc = align_up(sizeof(float) * n * nr, 256);
  const int64_t need = b_tok + b_ids + b_len + b_sc;
  if (need > h->io_cap) {
    PLLB_CUDA(cudaDeviceSynchronize());
    if (h->io) cudaFree(h->io);
    h->io = nullptr;
    h->io_cap = 0;
    PLLB_CUDA(cudaMalloc(&h->io, (size_t)need));
    h->io_cap = need;
  }
  uint8_t* base = reinterpret_cast<uint8_t*>(h->io);
  int32_t* d_tok = reinterpret_cast<int32_t*>(base);
  int32_t* d_ids = reinterpret_cast<int32_t*>(base + b_tok);
  int32_t* d_len = reinterpret_cast<int32_t*>(base + b_tok + b_ids);
  float* d_sc = reinterpret_cast<float*>(base + b_tok + b_ids + b_len);
  cudaStream_t s = 0;
  if (n_tok > 0) PLLB_CUDA(cudaMemcpyAsync(d_tok, tokens + off[0], sizeof(int32_t) * n_tok, cudaMemcpyHostToDevice, s));
  RC(generate_beam_impl(h, gen, beam, d_tok - off[0], off, n, d_ids, d_len, d_sc, s));
  PLLB_CUDA(cudaMemcpyAsync(out_ids, d_ids, sizeof(int32_t) * n * nr * ML, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaMemcpyAsync(out_len, d_len, sizeof(int32_t) * n * nr, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaMemcpyAsync(out_score, d_sc, sizeof(float) * n * nr, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  return PLLB_OK;
}

int pllb_s2s_debug_beam_replay(pllb_s2s h, const pllb_gen_desc* gen, const pllb_beam_desc* beam, int32_t n,
                               const float* hidden, int32_t steps, int32_t* out_ids, int32_t* out_len, float* out_score,
                               int32_t* out_parent, float* out_run_score) {
  if (!h) return fail(PLLB_ERR_INVALID, "null handle");
  RC(check_beam(h, gen, beam));
  const int K = gen->num_beams, ML = gen->max_length, H = h->d.hidden, nr = beam->num_return_sequences;
  if (n < 1 || (int64_t)n * K > h->max_rows) return fail(PLLB_ERR_INVALID, "replay: need 1 <= n * num_beams <= max_rows");
  if (steps != ML - 1) return fail(PLLB_ERR_INVALID, "replay: steps must be max_length - 1");
  if (!hidden || !out_ids || !out_len || !out_score || !out_parent || !out_run_score)
    return fail(PLLB_ERR_INVALID, "replay: null argument");
  PLLB_CUDA(cudaSetDevice(h->device));
  const int R = n * K;
  cudaStream_t s = 0;
  BeamState st{};
  float2* topk = nullptr;
  RC(beam_state(h, gen, beam, n, &st, &topk));
  RC(launch_beam_init(st, s));
  for (int64_t i = 0; i < (int64_t)steps * R; ++i) {
    out_parent[i] = -1;
    out_run_score[i] = 0.f;
  }
  for (int t = 1; t < ML; ++t) {
    PLLB_CUDA(cudaMemcpyAsync(h->enc_f32, hidden + (size_t)(t - 1) * R * H, sizeof(float) * R * H,
                              cudaMemcpyHostToDevice, s));
    RC(launch_f32_to_bf16(h->enc_f32, h->hid16, (int64_t)R * H, h->fp16, s));
    RC(beam_head_step(h, &st, topk, t, s));
    PLLB_CUDA(cudaMemcpyAsync(out_parent + (size_t)(t - 1) * R, st.parent, sizeof(int32_t) * R, cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaMemcpyAsync(out_run_score + (size_t)(t - 1) * R, st.run_score, sizeof(float) * R,
                              cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaMemcpyAsync(h->done_host, st.frozen_count, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    PLLB_CUDA(cudaStreamSynchronize(s));
    if (h->done_host[0] >= n) break;
  }
  int32_t* d_out = reinterpret_cast<int32_t*>(h->enc_f32);    // the hidden staging is free again
  int32_t* d_len = d_out + (size_t)n * nr * ML;
  float* d_sc = reinterpret_cast<float*>(d_len + (size_t)n * nr);
  RC(launch_beam_output(st, nr, d_out, d_len, d_sc, s));
  PLLB_CUDA(cudaMemcpyAsync(out_ids, d_out, sizeof(int32_t) * n * nr * ML, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaMemcpyAsync(out_len, d_len, sizeof(int32_t) * n * nr, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaMemcpyAsync(out_score, d_sc, sizeof(float) * n * nr, cudaMemcpyDeviceToHost, s));
  PLLB_CUDA(cudaStreamSynchronize(s));
  return PLLB_OK;
}

}  // extern "C"
