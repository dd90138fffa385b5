// seq2seq_kernels.cu — the small kernels of greedy encoder-decoder generation (pllb_generate).
//
// A decoder step over the rows in flight is: embedding + LayerNorm, then per layer the QKV GEMM,
// single-query self-attention over the row's KV cache, attention-output GEMM + LayerNorm, cross-Q
// GEMM, single-query cross-attention over the row's encoder K/V, output GEMM + LayerNorm and the
// FFN; then the LM head GEMM with the EPI_ARGMAX epilogue and argmax_finish.  The GEMMs are the
// tcgen05 kernels of gemm_tcgen05.cu / gemm_ln_tcgen05.cu; this file holds everything else.
// fp32 arithmetic, no atomics except the integer count of finished rows: a run is bit-deterministic.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>

#include "common.h"

namespace pllb {

namespace {

template <bool FP16>
__device__ __forceinline__ uint16_t to16(float x) {
  if constexpr (FP16) {                 // saturating, as the GEMM epilogues convert
    unsigned short h;
    asm("cvt.rn.f16.f32 %0, %1;" : "=h"(h) : "f"(fminf(fmaxf(x, -65504.f), 65504.f)));
    return h;
  }
  else return __bfloat16_as_ushort(__float2bfloat16_rn(x));
}
// two packed 16-bit values -> fp32 (low half first)
template <bool FP16>
__device__ __forceinline__ float2 unpack16x2(uint32_t w) {
  if constexpr (FP16) {
    float lo, hi;
    asm("{.reg .b16 l, h;\n mov.b32 {l, h}, %2;\n cvt.f32.f16 %0, l;\n cvt.f32.f16 %1, h;}"
        : "=f"(lo), "=f"(hi) : "r"(w));
    return make_float2(lo, hi);
  } else return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
// 8 consecutive 16-bit values (16-byte aligned) -> fp32
template <bool FP16>
__device__ __forceinline__ void ld16x8(const uint16_t* p, float* out) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  float2 f;
  f = unpack16x2<FP16>(u.x); out[0] = f.x; out[1] = f.y;
  f = unpack16x2<FP16>(u.y); out[2] = f.x; out[3] = f.y;
  f = unpack16x2<FP16>(u.z); out[4] = f.x; out[5] = f.y;
  f = unpack16x2<FP16>(u.w); out[6] = f.x; out[7] = f.y;
}

__global__ void decode_init_kernel(DecodeState st) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r == 0) *st.done_rows = 0;
  if (r >= st.rows) return;
  int32_t* ids = st.ids + (size_t)r * st.max_len;
  ids[0] = st.start_id;
  for (int j = 1; j < st.max_len; ++j) ids[j] = st.pad_id;
  if (st.logit)
    for (int j = 0; j < st.max_len; ++j) st.logit[(size_t)r * st.max_len + j] = 0.f;
  st.len[r] = 0;
  // the head launch of step 1 picks the forced BOS column (or the forced EOS one when max_len == 2)
  st.force_col[r] = st.max_len - 1 == 1 && st.forced_eos >= 0 ? st.forced_eos : st.forced_bos;
}

// One block of 256 threads per row; H <= 1024 (four columns per thread).
template <bool FP16>
__global__ void __launch_bounds__(256) dec_embed_kernel(DecodeState st, int pos, const float* __restrict__ word,
                                                        const float* __restrict__ pemb, const float* __restrict__ g,
                                                        const float* __restrict__ b, float eps, int H,
                                                        float* __restrict__ hid_f32, uint16_t* __restrict__ hid_16) {
  __shared__ float red[2][8];
  const int r = blockIdx.x;
  const int tok = st.ids[(size_t)r * st.max_len + pos];
  const float* wrow = word + (size_t)tok * H;
  const float* prow = pemb + (size_t)pos * H;
  float x[4];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = threadIdx.x + 256 * i;
    x[i] = c < H ? wrow[c] + prow[c] : 0.f;
    s += x[i];
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[0][warp] = s;
  __syncthreads();
  float mean = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) mean += red[0][w];
  mean /= (float)H;
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = threadIdx.x + 256 * i;
    const float d = c < H ? x[i] - mean : 0.f;
    v += d * d;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) red[1][warp] = v;
  __syncthreads();
  float var = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) var += red[1][w];
  const float rstd = rsqrtf(var / (float)H + eps);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int c = threadIdx.x + 256 * i;
    if (c < H) {
      const float y = (x[i] - mean) * rstd * g[c] + b[c];
      hid_f32[t32_index(r, c, H)] = y;
      hid_16[(size_t)r * H + c] = to16<FP16>(y);
    }
  }
}

// One warp per (row, head), four warps per block.  Lane j scores keys j, j + 32, ... (the full
// 64-wide query sits in registers, each key row is one 128-byte read); the softmax weights go
// through shared memory; for the weighted sum of V each lane owns two of the 64 dimensions.
template <bool FP16>
__global__ void __launch_bounds__(128, 4) decode_attention_kernel(
    const uint16_t* __restrict__ q, int q_stride, const uint16_t* kv, int64_t kv_stride,
    const int32_t* __restrict__ key_start, const int32_t* __restrict__ key_len, int self_t, int max_len,
    const uint16_t* __restrict__ new_kv, int new_kv_stride, uint16_t* kv_cache, uint16_t* __restrict__ ctx, int rows,
    int H, int NH, int max_keys) {
  extern __shared__ float sp[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t item = (int64_t)blockIdx.x * 4 + warp;
  if (item >= (int64_t)rows * NH) return;
  const int r = (int)(item / NH), h = (int)(item % NH);
  float* p = sp + warp * max_keys;
  const uint16_t* base;
  int64_t stride;
  int n;
  if (key_start == nullptr) {
    // self-attention: append this step's K | V (head h) to slot self_t of the row's cache, then read slots 0..t
    uint16_t* slot = kv_cache + ((size_t)r * max_len + self_t) * (size_t)(2 * H);
    const uint16_t* src = new_kv + (size_t)r * new_kv_stride;
    const int part = lane >> 4;                          // 0: K, 1: V
    const int c = h * 64 + (lane & 15) * 4;
    *reinterpret_cast<uint2*>(slot + part * H + c) = *reinterpret_cast<const uint2*>(src + part * H + c);
    __syncwarp();
    base = kv_cache + (size_t)r * max_len * (size_t)(2 * H);
    stride = 2 * H;
    n = self_t + 1;
  } else {
    base = kv + (size_t)key_start[r] * kv_stride;
    stride = kv_stride;
    n = key_len[r];
  }
  float qv[64];
  const uint16_t* qrow = q + (size_t)r * q_stride + h * 64;
#pragma unroll
  for (int i = 0; i < 8; ++i) ld16x8<FP16>(qrow + 8 * i, qv + 8 * i);
  float m = -INFINITY;
  for (int j = lane; j < n; j += 32) {
    const uint16_t* krow = base + (size_t)j * stride + h * 64;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float kf[8];
      ld16x8<FP16>(krow + 8 * i, kf);
#pragma unroll
      for (int e = 0; e < 8; ++e) acc = fmaf(qv[8 * i + e], kf[e], acc);
    }
    const float sc = acc * 0.125f;                       // head_dim ** -0.5
    p[j] = sc;
    m = fmaxf(m, sc);
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
  for (int j = lane; j < n; j += 32) {
    const float e = expf(p[j] - m);
    p[j] = e;
    sum += e;
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  __syncwarp();
  float o0 = 0.f, o1 = 0.f;
  const uint16_t* vcol = base + H + h * 64 + 2 * lane;
  for (int j = 0; j < n; ++j) {
    const float w = p[j];
    const uint32_t u = *reinterpret_cast<const uint32_t*>(vcol + (size_t)j * stride);
    const float2 v = unpack16x2<FP16>(u);
    o0 = fmaf(w, v.x, o0);
    o1 = fmaf(w, v.y, o1);
  }
  const float inv = 1.f / sum;
  const uint32_t packed = (uint32_t)to16<FP16>(o0 * inv) | ((uint32_t)to16<FP16>(o1 * inv) << 16);
  *reinterpret_cast<uint32_t*>(ctx + (size_t)r * H + h * 64 + 2 * lane) = packed;
}

__global__ void argmax_finish_kernel(const float2* __restrict__ parts, const float* __restrict__ forced_logit,
                                     int n_parts, DecodeState st, int t) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= st.rows) return;
  float best = -INFINITY;
  int arg = 0;
  const float2* pr = parts + (size_t)r * n_parts;
  for (int i = 0; i < n_parts; ++i) {              // parts ascend in column: strict > keeps the first maximum
    const float2 v = pr[i];
    if (v.x > best || i == 0) { best = v.x; arg = __float_as_int(v.y); }
  }
  const int forced = t == st.max_len - 1 && st.forced_eos >= 0 ? st.forced_eos : t == 1 ? st.forced_bos : -1;
  if (forced >= 0) { arg = forced; best = forced_logit[r]; }
  const bool finished = st.len[r] > 0;
  int tok = arg;
  float lg = best;
  if (finished) { tok = st.pad_id; lg = 0.f; }
  st.ids[(size_t)r * st.max_len + t] = tok;
  if (st.logit) st.logit[(size_t)r * st.max_len + t] = lg;
  if (!finished && (tok == st.eos_id || t == st.max_len - 1)) {
    st.len[r] = t + 1;
    if (tok == st.eos_id) atomicAdd(st.done_rows, 1);
  }
  // the column the next step's head launch picks
  const int tn = t + 1;
  st.force_col[r] = tn == st.max_len - 1 && st.forced_eos >= 0 ? st.forced_eos : tn == 1 ? st.forced_bos : -1;
}

__global__ void scale_copy_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t n, float scale) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[i] * scale;
}

}  // namespace

int launch_decode_init(DecodeState st, cudaStream_t s) {
  decode_init_kernel<<<(unsigned)ceil_div(std::max(st.rows, 1), 256), 256, 0, s>>>(st);
  PLLB_LAUNCH_CHECK("decode_init_kernel");
  return PLLB_OK;
}

int launch_dec_embed(const DecodeState& st, int pos, const float* word_scaled, const float* pos_emb, const float* g,
                     const float* b, float eps, int H, float* hid_f32, void* hid_16, bool fp16, cudaStream_t s) {
  if (st.rows <= 0) return PLLB_OK;
  if (H > 1024) return fail(PLLB_ERR_INVALID, "dec_embed: hidden > 1024");
  uint16_t* o16 = reinterpret_cast<uint16_t*>(hid_16);
  if (fp16) dec_embed_kernel<true><<<st.rows, 256, 0, s>>>(st, pos, word_scaled, pos_emb, g, b, eps, H, hid_f32, o16);
  else dec_embed_kernel<false><<<st.rows, 256, 0, s>>>(st, pos, word_scaled, pos_emb, g, b, eps, H, hid_f32, o16);
  PLLB_LAUNCH_CHECK("dec_embed_kernel");
  return PLLB_OK;
}

int launch_decode_attention(const void* q, int q_stride, const void* kv, int64_t kv_stride, const int32_t* key_start,
                            const int32_t* key_len, int self_t, int max_len, const void* new_kv, int new_kv_stride,
                            void* kv_cache, void* ctx, int rows, int H, int max_keys, bool fp16, cudaStream_t s) {
  if (rows <= 0) return PLLB_OK;
  const int NH = H / 64;
  const int64_t items = (int64_t)rows * NH;
  const unsigned grid = (unsigned)ceil_div(items, 4);
  const size_t smem = (size_t)4 * std::max(max_keys, 1) * sizeof(float);
  if (smem > 48 * 1024) return fail(PLLB_ERR_INVALID, "decode_attention: more than 3072 keys");
  auto* qq = reinterpret_cast<const uint16_t*>(q);
  auto* kk = reinterpret_cast<const uint16_t*>(kv);
  auto* nk = reinterpret_cast<const uint16_t*>(new_kv);
  auto* kc = reinterpret_cast<uint16_t*>(kv_cache);
  auto* cc = reinterpret_cast<uint16_t*>(ctx);
  if (fp16)
    decode_attention_kernel<true><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len, self_t, max_len,
                                                          nk, new_kv_stride, kc, cc, rows, H, NH, max_keys);
  else
    decode_attention_kernel<false><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len, self_t,
                                                           max_len, nk, new_kv_stride, kc, cc, rows, H, NH, max_keys);
  PLLB_LAUNCH_CHECK("decode_attention_kernel");
  return PLLB_OK;
}

int launch_argmax_finish(const float2* partials, const float* forced_logit, int n_parts, DecodeState st, int t,
                         cudaStream_t s) {
  if (st.rows <= 0) return PLLB_OK;
  argmax_finish_kernel<<<(unsigned)ceil_div(st.rows, 128), 128, 0, s>>>(partials, forced_logit, n_parts, st, t);
  PLLB_LAUNCH_CHECK("argmax_finish_kernel");
  return PLLB_OK;
}

int launch_scale_copy(const float* src, float* dst, int64_t n, float scale, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  const int64_t blocks = std::min<int64_t>(ceil_div(n, 256), 4096);
  scale_copy_kernel<<<(unsigned)blocks, 256, 0, s>>>(src, dst, n, scale);
  PLLB_LAUNCH_CHECK("scale_copy_kernel");
  return PLLB_OK;
}

}  // namespace pllb
