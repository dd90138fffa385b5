// train_kernels.cu — the non-GEMM kernels of the MLM fine-tuning path (MLM_PLL/main.py:73-99 with
// train_mode=True; transformers BertForMaskedLM forward with labels + autograd + torch.optim.AdamW
// in the reference).  The matrix products (forward, dgrad, wgrad) all run on the tcgen05 GEMM of
// gemm_tcgen05.cu, which multiplies two K-contiguous 16-bit operands: the kernels here produce the
// row-major and the transposed 16-bit copies it needs, and everything that is not a GEMM —
// embeddings, LayerNorm forward / backward with saved statistics, GELU, the padded-batch attention
// forward and its two backward passes, the all-position cross entropy, bias and LayerNorm
// parameter gradients, the embedding scatter, AdamW.  A training batch is B zero-padded sequences
// of T rows (the reference's collate, MLM_PLL/main.py:28-54): pad rows are real rows (input id 0,
// label 0) that attend to the n_valid[b] real keys and contribute to the loss, as in the reference.
// Every reduction runs in a fixed order (no floating-point atomics): a step is deterministic.
#include <cuda_bf16.h>

#include <algorithm>
#include <cmath>

#include "common.h"
#include "train.h"

namespace pllb {
namespace {

constexpr int RW = 4;   // warps (= rows) per block of the row kernels

__device__ __forceinline__ float wsum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Stateless dropout: element `idx` of site `site` is kept iff a 64-bit mix of (seed, site, idx)
// is >= thresh (drop probability thresh / 2^32); kept elements are scaled by 1 / (1 - p).  The
// backward pass regenerates the same mask, nothing is stored.
__device__ __forceinline__ float drop_factor(const TrainDrop& d, uint32_t site, uint64_t idx) {
  if (d.thresh == 0) return 1.f;
  uint64_t x = __ldg(d.seed) + (uint64_t)site * 0x9E3779B97F4A7C15ull + idx * 0xD1B54A32D192ED03ull;
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return (uint32_t)(x >> 32) >= d.thresh ? d.inv_keep : 0.f;
}

__device__ __forceinline__ float gelu_exact(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float gelu_grad(float x) {
  return 0.5f * (1.f + erff(x * 0.70710678118654752f)) + x * 0.3989422804014327f * __expf(-0.5f * x * x);
}

// ---------------------------------------------------------------- LayerNorm forward (row per warp)
// z = drop(y) + res  (res may be null; EMBED: z = word[id] + pos[r % T] + type[0], dropout AFTER the
// LayerNorm as in BertEmbeddings);  out = LN(z);  saves xhat and rstd for the backward pass.
template <int NV, bool EMBED>
__global__ void __launch_bounds__(RW * 32)
ln_fwd_kernel(const float* __restrict__ y, const float* res, const int32_t* __restrict__ ids, int T,
              const float* __restrict__ word, const float* __restrict__ pos, const float* __restrict__ type,
              const float* __restrict__ g, const float* __restrict__ b, float eps, int R, TrainDrop drop, uint32_t site,
              float* out32, __nv_bfloat16* __restrict__ out16, float* __restrict__ xhat, float* __restrict__ rstd) {
  constexpr int H = NV * 32;
  const int r = blockIdx.x * RW + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
  float v[NV];
  float s = 0.f;
  if (EMBED) {
    const int id = ids[r], p = r % T;
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      v[i] = word[(size_t)id * H + c] + type[c] + pos[(size_t)p * H + c];
      s += v[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int c = lane + 32 * i;
      const size_t e = (size_t)r * H + c;
      v[i] = y[e] * drop_factor(drop, site, e) + (res ? res[e] : 0.f);
      s += v[i];
    }
  }
  const float mean = wsum(s) * (1.f / H);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { const float d = v[i] - mean; q += d * d; }
  const float rs = rsqrtf(wsum(q) * (1.f / H) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    const size_t e = (size_t)r * H + c;
    const float xh = (v[i] - mean) * rs;
    float o = xh * g[c] + b[c];
    if (EMBED) o *= drop_factor(drop, site, e);
    if (xhat) xhat[e] = xh;
    if (out32) out32[e] = o;
    if (out16) out16[e] = __float2bfloat16_rn(o);
  }
  if (lane == 0 && rstd) rstd[r] = rs;
}

// ---------------------------------------------------------------- LayerNorm backward (row per warp)
// dy_tot = (dy + add) * [drop_in]   (written back to dy: the parameter-gradient kernel reads it)
// dz     = rstd * (dxh - mean(dxh) - xhat * mean(dxh * xhat)),  dxh = dy_tot * gamma
// dz_drop = dz * [drop_out]         (gradient of the GEMM output that went through dropout)
template <int NV>
__global__ void __launch_bounds__(RW * 32)
ln_bwd_kernel(float* dy, const float* add, const float* __restrict__ g, const float* __restrict__ xhat,
              const float* __restrict__ rstd, int R, TrainDrop drop, int site_in, int site_out, float* dz, float* dz_drop) {
  constexpr int H = NV * 32;
  const int r = blockIdx.x * RW + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
  // all loads first, all stores last: dy / add / dz may alias, so a store inside the load loop would
  // serialise the iterations on the memory latency (measured: 20 us instead of 5 for 643 rows)
  float d[NV], xh[NV], t[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const size_t e = (size_t)r * H + lane + 32 * i;
    t[i] = dy[e] + (add ? add[e] : 0.f);
    xh[i] = xhat[e];
  }
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    if (site_in >= 0) t[i] *= drop_factor(drop, (uint32_t)site_in, (size_t)r * H + c);
    d[i] = t[i] * g[c];
    s1 += d[i];
    s2 += d[i] * xh[i];
  }
  const float m1 = wsum(s1) * (1.f / H), m2 = wsum(s2) * (1.f / H), rs = rstd[r];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const size_t e = (size_t)r * H + lane + 32 * i;
    const float z = rs * (d[i] - m1 - xh[i] * m2);
    dy[e] = t[i];
    dz[e] = z;
    if (dz_drop) dz_drop[e] = site_out >= 0 ? z * drop_factor(drop, (uint32_t)site_out, e) : z;
  }
}

// dgamma[c] = sum_r dy[r,c] * xhat[r,c], dbeta[c] = sum_r dy[r,c]; also the plain column sum (bias
// gradients; xhat == nullptr).  Block = 32 columns x 8 row groups over the row slice
// [blockIdx.y * rows_per_split, ...); with gridDim.y > 1 the per-slice sums go to `part` ([S, 2, C]) and
// colsum_final_kernel adds the slices in order — a fixed summation order, so deterministic.
template <typename TIn>
__global__ void __launch_bounds__(256)
colsum_kernel(const TIn* __restrict__ dy, const float* __restrict__ xhat, int R, int C, int rows_per_split,
              float* __restrict__ out_sum, float* __restrict__ out_dot, float* __restrict__ part) {
  __shared__ float s_sum[8][33], s_dot[8][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + tx;
  const int r_begin = blockIdx.y * rows_per_split, r_end = min(R, r_begin + rows_per_split);
  float a = 0.f, d = 0.f;
  if (c < C) {
#pragma unroll 4
    for (int r = r_begin + ty; r < r_end; r += 8) {
      const size_t e = (size_t)r * C + c;
      float v;
      if constexpr (sizeof(TIn) == 2) v = __bfloat162float(dy[e]); else v = dy[e];
      a += v;
      if (xhat) d += v * xhat[e];
    }
  }
  s_sum[ty][tx] = a;
  s_dot[ty][tx] = d;
  __syncthreads();
  if (ty == 0 && c < C) {
    float sa = 0.f, sd = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) { sa += s_sum[k][tx]; sd += s_dot[k][tx]; }
    if (gridDim.y > 1) {
      part[((size_t)blockIdx.y * 2) * C + c] = sa;
      part[((size_t)blockIdx.y * 2 + 1) * C + c] = sd;
    } else {
      if (out_sum) out_sum[c] = sa;
      if (out_dot) out_dot[c] = sd;
    }
  }
}
__global__ void colsum_final_kernel(const float* __restrict__ part, int S, int C, float* __restrict__ out_sum,
                                    float* __restrict__ out_dot) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float sa = 0.f, sd = 0.f;
  for (int k = 0; k < S; ++k) { sa += part[((size_t)k * 2) * C + c]; sd += part[((size_t)k * 2 + 1) * C + c]; }
  if (out_sum) out_sum[c] = sa;
  if (out_dot) out_dot[c] = sd;
}

// ---------------------------------------------------------------- GELU
__global__ void gelu_fwd_kernel(const float* __restrict__ f, int64_t n, __nv_bfloat16* __restrict__ out16,
                                float* __restrict__ out32) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = gelu_exact(f[i]);
    if (out16) out16[i] = __float2bfloat16_rn(v);
    if (out32) out32[i] = v;
  }
}
__global__ void gelu_bwd_kernel(float* __restrict__ dg, const float* __restrict__ f, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dg[i] *= gelu_grad(f[i]);
}

// ---------------------------------------------------------------- 16-bit copies for the GEMMs
// src [R, C] (fp32 or bf16) -> dst16 [R, C] (optional) and dstT [C, Rp] (optional; columns r >= R are 0).
// 32 x 32 tiles through shared memory; block (32, 8).
template <typename TIn>
__global__ void __launch_bounds__(256)
cast_transpose_kernel(const TIn* __restrict__ src, int R, int C, int Rp, __nv_bfloat16* __restrict__ dst16,
                      __nv_bfloat16* __restrict__ dstT) {
  __shared__ __nv_bfloat16 tile[32][34];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = r0 + ty + 8 * k, c = c0 + tx;
    __nv_bfloat16 v = __float2bfloat16_rn(0.f);
    if (r < R && c < C) {
      if constexpr (sizeof(TIn) == 2) v = src[(size_t)r * C + c]; else v = __float2bfloat16_rn(src[(size_t)r * C + c]);
      if (dst16) dst16[(size_t)r * C + c] = v;
    }
    tile[ty + 8 * k][tx] = v;
  }
  __syncthreads();
  if (!dstT) return;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = c0 + ty + 8 * k, r = r0 + tx;
    if (c < C && r < Rp) dstT[(size_t)c * Rp + r] = tile[tx][ty + 8 * k];
  }
}

// ---------------------------------------------------------------- attention (padded batch), warp per (row, head)
__device__ __forceinline__ float dot64_bf16(const float* __restrict__ a /* smem, 64 floats */,
                                            const __nv_bfloat16* __restrict__ b /* 64 contiguous bf16 */) {
  float s = 0.f;
  const uint4* p = reinterpret_cast<const uint4*>(b);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const uint4 u = p[k];
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[j]));
      s += a[k * 8 + 2 * j] * f.x + a[k * 8 + 2 * j + 1] * f.y;
    }
  }
  return s;
}
__device__ __forceinline__ float dot64_f32(const float* __restrict__ a /* smem */, const float* __restrict__ b /* global */) {
  float s = 0.f;
  const float4* p = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float4 u = p[k];
    s += a[4 * k] * u.x + a[4 * k + 1] * u.y + a[4 * k + 2] * u.z + a[4 * k + 3] * u.w;
  }
  return s;
}

// ctx[r, h*64 + d] = sum_j drop(softmax_j(q_r . k_j / 8)) * v_j[d] over the n_valid keys of r's sequence
__global__ void __launch_bounds__(RW * 32)
attn_fwd_train_kernel(const __nv_bfloat16* __restrict__ qkv, const int32_t* __restrict__ n_valid, int R, int T, int H, int NH,
                      TrainDrop drop, uint32_t site, __nv_bfloat16* __restrict__ ctx, float* __restrict__ lse_out) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= R * NH) return;
  const int r = item / NH, h = item % NH, seq = r / T, i = r % T, nv = n_valid[seq];
  float* sq = smem + (size_t)w * (64 + T);
  float* sp = sq + 64;
  const size_t ld = (size_t)3 * H;
  const __nv_bfloat16* base = qkv + (size_t)seq * T * ld + (size_t)h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)i * ld + 2 * lane));
    sq[2 * lane] = f.x; sq[2 * lane + 1] = f.y;
  }
  __syncwarp();
  float m = -INFINITY;
  for (int j = lane; j < nv; j += 32) {
    const float s = dot64_bf16(sq, base + (size_t)j * ld + H) * 0.125f;
    sp[j] = s;
    m = fmaxf(m, s);
  }
  m = wmax(m);
  float l = 0.f;
  for (int j = lane; j < nv; j += 32) l += __expf(sp[j] - m);
  const float lse = m + __logf(wsum(l));
  const uint64_t pbase = ((uint64_t)(seq * NH + h) * T + i) * T;
  for (int j = lane; j < nv; j += 32) sp[j] = __expf(sp[j] - lse) * drop_factor(drop, site, pbase + j);
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
  for (int j = 0; j < nv; ++j) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)j * ld + 2 * H + 2 * lane));
    a0 += sp[j] * f.x; a1 += sp[j] * f.y;
  }
  *reinterpret_cast<__nv_bfloat162*>(ctx + (size_t)r * H + h * 64 + 2 * lane) = __floats2bfloat162_rn(a0, a1);
  if (lane == 0) lse_out[item] = lse;
}

// dq of row r (and D_r = sum_j P_rj dP_rj, kept for the dk / dv pass)
__global__ void __launch_bounds__(RW * 32)
attn_bwd_q_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ dctx, const float* __restrict__ lse,
                  const int32_t* __restrict__ n_valid, int R, int T, int H, int NH, TrainDrop drop, uint32_t site,
                  float* __restrict__ dqkv, float* __restrict__ Dout) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= R * NH) return;
  const int r = item / NH, h = item % NH, seq = r / T, i = r % T, nv = n_valid[seq];
  float* sq = smem + (size_t)w * (128 + 2 * T);
  float* sdo = sq + 64;
  float* sp = sdo + 64;
  float* sds = sp + T;
  const size_t ld = (size_t)3 * H;
  const __nv_bfloat16* base = qkv + (size_t)seq * T * ld + (size_t)h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)i * ld + 2 * lane));
    sq[2 * lane] = f.x; sq[2 * lane + 1] = f.y;
    const float2 g = *reinterpret_cast<const float2*>(dctx + (size_t)r * H + h * 64 + 2 * lane);
    sdo[2 * lane] = g.x; sdo[2 * lane + 1] = g.y;
  }
  __syncwarp();
  const float ls = lse[item];
  const uint64_t pbase = ((uint64_t)(seq * NH + h) * T + i) * T;
  float dpart = 0.f;
  for (int j = lane; j < nv; j += 32) {
    const float p = __expf(dot64_bf16(sq, base + (size_t)j * ld + H) * 0.125f - ls);
    const float dp = dot64_bf16(sdo, base + (size_t)j * ld + 2 * H) * drop_factor(drop, site, pbase + j);
    sp[j] = p; sds[j] = dp;
    dpart += p * dp;
  }
  const float D = wsum(dpart);
  for (int j = lane; j < nv; j += 32) sds[j] = sp[j] * (sds[j] - D);
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
  for (int j = 0; j < nv; ++j) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)j * ld + H + 2 * lane));
    a0 += sds[j] * f.x; a1 += sds[j] * f.y;
  }
  *reinterpret_cast<float2*>(dqkv + (size_t)r * ld + h * 64 + 2 * lane) = make_float2(a0 * 0.125f, a1 * 0.125f);
  if (lane == 0) Dout[item] = D;
}

// dk and dv of key row r: sums over ALL T query rows of the sequence (pad queries included)
__global__ void __launch_bounds__(RW * 32)
attn_bwd_kv_kernel(const __nv_bfloat16* __restrict__ qkv, const float* __restrict__ dctx, const float* __restrict__ lse,
                   const float* __restrict__ Dq, const int32_t* __restrict__ n_valid, int R, int T, int H, int NH,
                   TrainDrop drop, uint32_t site, float* __restrict__ dqkv) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= R * NH) return;
  const int r = item / NH, h = item % NH, seq = r / T, j = r % T, nv = n_valid[seq];
  const size_t ld = (size_t)3 * H;
  float2* dk_out = reinterpret_cast<float2*>(dqkv + (size_t)r * ld + H + h * 64 + 2 * lane);
  float2* dv_out = reinterpret_cast<float2*>(dqkv + (size_t)r * ld + 2 * H + h * 64 + 2 * lane);
  if (j >= nv) {                       // a masked key: probability 0 for every query
    *dk_out = make_float2(0.f, 0.f);
    *dv_out = make_float2(0.f, 0.f);
    return;
  }
  float* sk = smem + (size_t)w * (128 + 2 * T);
  float* sv = sk + 64;
  float* sds = sv + 64;
  float* spd = sds + T;
  const __nv_bfloat16* base = qkv + (size_t)seq * T * ld + (size_t)h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)j * ld + H + 2 * lane));
    sk[2 * lane] = f.x; sk[2 * lane + 1] = f.y;
    const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)j * ld + 2 * H + 2 * lane));
    sv[2 * lane] = g.x; sv[2 * lane + 1] = g.y;
  }
  __syncwarp();
  for (int i = lane; i < T; i += 32) {
    const int ri = seq * T + i;
    const float p = __expf(dot64_bf16(sk, base + (size_t)i * ld) * 0.125f - lse[(size_t)ri * NH + h]);
    const float sc = drop_factor(drop, site, ((uint64_t)(seq * NH + h) * T + i) * T + j);
    const float dp = dot64_f32(sv, dctx + (size_t)ri * H + h * 64) * sc;
    sds[i] = p * (dp - Dq[(size_t)ri * NH + h]);
    spd[i] = p * sc;
  }
  __syncwarp();
  float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
#pragma unroll 4
  for (int i = 0; i < T; ++i) {
    const int ri = seq * T + i;
    const float2 q = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(base + (size_t)i * ld + 2 * lane));
    const float2 g = *reinterpret_cast<const float2*>(dctx + (size_t)ri * H + h * 64 + 2 * lane);
    k0 += sds[i] * q.x; k1 += sds[i] * q.y;
    v0 += spd[i] * g.x; v1 += spd[i] * g.y;
  }
  *dk_out = make_float2(k0 * 0.125f, k1 * 0.125f);
  *dv_out = make_float2(v0, v1);
}

// ---------------------------------------------------------------- cross entropy over every position
// loss_r = logsumexp(logits[r, :V]) - logits[r, label_r];  dlogits = softmax - onehot (bf16, UNSCALED: the
// -1 of the label column stays exact; with the 1/R of the mean folded in, every one-hot entry would
// carry the same bf16 rounding error of 1/R — a systematic scale error of up to 0.4 % on every
// gradient.  The consumers multiply by 1/R in fp32.)
__global__ void __launch_bounds__(256)
ce_kernel(const float* __restrict__ logits, const int32_t* __restrict__ labels, int V, int Vp,
          float* __restrict__ loss_rows, __nv_bfloat16* __restrict__ dlogits) {
  __shared__ float red[8];
  __shared__ float bc;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const float* x = logits + (size_t)r * Vp;
  float m = -INFINITY;
  for (int c = tid; c < V; c += 256) m = fmaxf(m, x[c]);
  m = wmax(m);
  if (lane == 0) red[w] = m;
  __syncthreads();
  if (tid == 0) { float t = red[0]; for (int k = 1; k < 8; ++k) t = fmaxf(t, red[k]); bc = t; }
  __syncthreads();
  m = bc;
  float s = 0.f;
  for (int c = tid; c < V; c += 256) s += __expf(x[c] - m);
  s = wsum(s);
  __syncthreads();
  if (lane == 0) red[w] = s;
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int k = 0; k < 8; ++k) t += red[k]; bc = m + logf(t); }
  __syncthreads();
  const float lse = bc;
  const int label = labels[r];
  if (tid == 0) loss_rows[r] = lse - x[label];
  if (dlogits) {
    __nv_bfloat16* d = dlogits + (size_t)r * Vp;
    for (int c = tid; c < Vp; c += 256) {
      float g = 0.f;
      if (c < V) g = __expf(x[c] - lse) - (c == label ? 1.f : 0.f);
      d[c] = __float2bfloat16_rn(g);
    }
  }
}

__global__ void scale_kernel(float* __restrict__ x, int64_t n, float alpha) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= alpha;
}

// mean of the R per-row losses in a fixed order (double accumulation); single block
__global__ void __launch_bounds__(256) loss_mean_kernel(const float* __restrict__ loss_rows, int R, float* __restrict__ out) {
  __shared__ double red[256];
  double a = 0.0;
  for (int r = threadIdx.x; r < R; r += 256) a += (double)loss_rows[r];
  red[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[0] = (float)(red[0] / (double)R);
}

// ---------------------------------------------------------------- embedding gradients
// position rows: dpos[p, c] = sum_b dz[b*T + p, c] for p < T, 0 for the rows no batch row maps to
__global__ void pos_grad_kernel(const float* __restrict__ dz, int B, int T, int H, int max_pos, float* __restrict__ dpos) {
  const int64_t n = (int64_t)max_pos * H;
  for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(e / H), c = (int)(e % H);
    float a = 0.f;
    if (p < T)
      for (int b = 0; b < B; ++b) a += dz[((size_t)b * T + p) * H + c];
    dpos[e] = a;
  }
}
// word rows: the first row holding an id adds the rows of all its occurrences, in order, to dword[id]
// (which already holds the tied decoder's gradient).  The lookup sends nothing to the padding row
// (nn.Embedding(padding_idx = pad_token_id), transformers modeling_bert.py:75).
__global__ void __launch_bounds__(256)
word_grad_kernel(const float* __restrict__ dz, const int32_t* __restrict__ ids, int R, int H, int pad_id,
                 float* __restrict__ dword) {
  __shared__ int dup;
  const int r = blockIdx.x, id = ids[r];
  if (id == pad_id) return;
  if (threadIdx.x == 0) dup = 0;
  __syncthreads();
  for (int k = threadIdx.x; k < r; k += 256)
    if (ids[k] == id) dup = 1;
  __syncthreads();
  if (dup) return;
  for (int c = threadIdx.x; c < H; c += 256) {
    float a = 0.f;
    for (int k = r; k < R; ++k)
      if (ids[k] == id) a += dz[(size_t)k * H + c];
    dword[(size_t)id * H + c] += a;
  }
}

// ---------------------------------------------------------------- AdamW (torch.optim.AdamW, single-tensor path)
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                             int64_t n, float lr, float beta1, float beta2, float eps, float wd,
                             const TrainStepParams* __restrict__ scalars) {
  const float step_size = scalars->adam_step_size, bc2_sqrt = scalars->adam_bc2_sqrt;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float pi = p[i] * (1.f - lr * wd);
    const float gi = g[i];
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
    const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - step_size * (mi / denom);
  }
}

// ---------------------------------------------------------------- RescoreBert head (sequence score of the [CLS] row)
// s_b = linear_w . h[b*T, :] + linear_b; a warp per hypothesis, lane-strided fp32 sums then a fixed butterfly
template <int NV>
__global__ void __launch_bounds__(RW * 32)
cls_fwd_kernel(const float* __restrict__ h, const float* __restrict__ w, const float* __restrict__ bias, int B, int T,
               float* __restrict__ scores) {
  constexpr int H = NV * 32;
  const int b = blockIdx.x * RW + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* x = h + (size_t)b * T * H;
  float a = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) a += x[lane + 32 * i] * w[lane + 32 * i];
  a = wsum(a);
  if (lane == 0) scores[b] = a + bias[0];
}

// Loss over the B scores, one CTA.  Rows of a group are contiguous and group[] numbers them 0, 1, ...
// (checked on the host), so G = group[B-1] + 1 and one captured graph serves every grouping of B rows.
//   MD:   L_MD = (1/B) sum_i (s_i - y_i)^2,                         dL_MD/ds_i = (2/B) (s_i - y_i)
//   MWER: P = softmax_g(am_weight * a + s),  L_MWER = (1/G) sum_g sum_{i in g} P_i (e_i - mean_g e),
//         dL_MWER/ds_i = (1/G) P_i (e_i - sum_{j in g} P_j e_j)
// The thread that owns the first row of a group walks the whole group in row order; the loss sums run
// in double over a fixed tree.  dscore (fp32, the 1/B and 1/G already applied) is written when non-null.
__global__ void __launch_bounds__(256)
cls_loss_kernel(const float* __restrict__ scores, const float* __restrict__ target, const float* __restrict__ am,
                const float* __restrict__ err, const int32_t* __restrict__ group, int B, float md_weight, float mwer_weight,
                float am_weight, float* __restrict__ dscore, float* __restrict__ out_loss) {
  __shared__ double red_md[256], red_mw[256];
  const int tid = threadIdx.x;
  const int G = group[B - 1] + 1;
  const float inv_b = 1.f / (float)B, inv_g = 1.f / (float)G;
  double md = 0.0, mw = 0.0;
  for (int i = tid; i < B; i += 256) {
    const float d = scores[i] - target[i];
    md += (double)d * (double)d;
    if (dscore) dscore[i] = md_weight * (2.f * inv_b) * d;
  }
  __syncthreads();      // every dscore[i] holds its MD part before the group walks add to it
  if (mwer_weight != 0.f) {
    for (int i = tid; i < B; i += 256) {
      if (i > 0 && group[i] == group[i - 1]) continue;
      int end = i + 1;
      while (end < B && group[end] == group[i]) ++end;
      float m = -INFINITY;
      for (int j = i; j < end; ++j) m = fmaxf(m, am_weight * am[j] + scores[j]);
      float z = 0.f, pe = 0.f, es = 0.f;
      for (int j = i; j < end; ++j) {
        const float p = __expf(am_weight * am[j] + scores[j] - m);
        z += p;
        pe += p * err[j];
        es += err[j];
      }
      const float inv_z = 1.f / z, ebar_p = pe * inv_z, ebar = es / (float)(end - i);
      float lg = 0.f;
      for (int j = i; j < end; ++j) {
        const float p = __expf(am_weight * am[j] + scores[j] - m) * inv_z;
        lg += p * (err[j] - ebar);
        if (dscore) dscore[j] += mwer_weight * inv_g * p * (err[j] - ebar_p);
      }
      mw += (double)lg;
    }
  }
  red_md[tid] = md;
  red_mw[tid] = mw;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) { red_md[tid] += red_md[tid + o]; red_mw[tid] += red_mw[tid + o]; }
    __syncthreads();
  }
  if (tid == 0) out_loss[0] = (float)((double)md_weight * red_md[0] / (double)B + (double)mwer_weight * red_mw[0] / (double)G);
}

// Backward of the head.  Block 0: dlinear_w[c] = sum_b dscore_b * h[b*T, c], dlinear_b = sum_b dscore_b (row
// order).  Blocks >= 1: the top-layer gradient dh [R, H], zero except row b*T = dscore_b * linear_w.
__global__ void __launch_bounds__(256)
cls_bwd_kernel(const float* __restrict__ h, const float* __restrict__ w, const float* __restrict__ dscore, int B, int T,
               int H, float* __restrict__ dw, float* __restrict__ db, float* __restrict__ dh) {
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < H; c += blockDim.x) {
      float a = 0.f;
      for (int b = 0; b < B; ++b) a += dscore[b] * h[(size_t)b * T * H + c];
      dw[c] = a;
    }
    if (threadIdx.x == 0) {
      float a = 0.f;
      for (int b = 0; b < B; ++b) a += dscore[b];
      db[0] = a;
    }
    return;
  }
  const int64_t n = (int64_t)B * T * H;
  for (int64_t e = (blockIdx.x - 1) * (int64_t)blockDim.x + threadIdx.x; e < n; e += (int64_t)(gridDim.x - 1) * blockDim.x) {
    const int64_t r = e / H;
    const int c = (int)(e % H);
    dh[e] = r % T == 0 ? dscore[r / T] * w[c] : 0.f;
  }
}

int grid_for(int64_t n, int block) { return (int)std::min<int64_t>(ceil_div(n, block), 148 * 16); }

}  // namespace

// ================================================================== launchers
#define DISPATCH_NV(H, ...)                                    \
  switch ((H) / 32) {                                          \
    case 8:  { constexpr int NV = 8;  __VA_ARGS__; } break;    \
    case 16: { constexpr int NV = 16; __VA_ARGS__; } break;    \
    case 24: { constexpr int NV = 24; __VA_ARGS__; } break;    \
    case 32: { constexpr int NV = 32; __VA_ARGS__; } break;    \
    default: return fail(PLLB_ERR_INVALID, "train: hidden must be 256, 512, 768 or 1024"); \
  }

int launch_train_embed(const int32_t* ids, int T, const float* word, const float* pos, const float* type, const float* g,
                       const float* b, float eps, int R, int H, TrainDrop drop, uint32_t site, float* out32, void* out16,
                       float* xhat, float* rstd, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const int grid = (int)ceil_div(R, RW);
  DISPATCH_NV(H, ln_fwd_kernel<NV, true><<<grid, RW * 32, 0, s>>>(nullptr, nullptr, ids, T, word, pos, type, g, b, eps, R, drop,
                                                                  site, out32, reinterpret_cast<__nv_bfloat16*>(out16), xhat, rstd));
  PLLB_LAUNCH_CHECK("ln_fwd_kernel<embed>");
  return PLLB_OK;
}

int launch_train_ln_fwd(const float* y, const float* res, const float* g, const float* b, float eps, int R, int H,
                        TrainDrop drop, uint32_t site, float* out32, void* out16, float* xhat, float* rstd, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const int grid = (int)ceil_div(R, RW);
  DISPATCH_NV(H, ln_fwd_kernel<NV, false><<<grid, RW * 32, 0, s>>>(y, res, nullptr, 1, nullptr, nullptr, nullptr, g, b, eps, R,
                                                                   drop, site, out32, reinterpret_cast<__nv_bfloat16*>(out16), xhat, rstd));
  PLLB_LAUNCH_CHECK("ln_fwd_kernel");
  return PLLB_OK;
}

int launch_train_ln_bwd(float* dy, const float* add, const float* g, const float* xhat, const float* rstd, int R, int H,
                        TrainDrop drop, int site_in, int site_out, float* dz, float* dz_drop, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const int grid = (int)ceil_div(R, RW);
  DISPATCH_NV(H, ln_bwd_kernel<NV><<<grid, RW * 32, 0, s>>>(dy, add, g, xhat, rstd, R, drop, site_in, site_out, dz, dz_drop));
  PLLB_LAUNCH_CHECK("ln_bwd_kernel");
  return PLLB_OK;
}

int launch_train_colsum(const void* dy, bool dy_bf16, const float* xhat, int R, int C, float* out_sum, float* out_dot,
                        float* scratch, cudaStream_t s) {
  if (C <= 0) return PLLB_OK;
  // row slices of >= 64 rows, at most TRAIN_COLSUM_SPLITS of them, enough blocks to cover the chip
  int S = scratch ? (int)std::min<int64_t>(TRAIN_COLSUM_SPLITS, ceil_div(R, 64)) : 1;
  S = std::max(1, std::min<int>(S, (int)ceil_div(8 * 148, ceil_div(C, 32))));    // 8 resident blocks of 256 threads per SM
  const int rows_per_split = (int)ceil_div(std::max(R, 1), S);
  dim3 grid((unsigned)ceil_div(C, 32), (unsigned)S);
  if (dy_bf16) colsum_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(dy), xhat, R, C, rows_per_split, out_sum, out_dot, scratch);
  else colsum_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(dy), xhat, R, C, rows_per_split, out_sum, out_dot, scratch);
  PLLB_LAUNCH_CHECK("colsum_kernel");
  if (S > 1) {
    colsum_final_kernel<<<(int)ceil_div(C, 256), 256, 0, s>>>(scratch, S, C, out_sum, out_dot);
    PLLB_LAUNCH_CHECK("colsum_final_kernel");
  }
  return PLLB_OK;
}

int launch_train_gelu_fwd(const float* f, int64_t n, void* out16, float* out32, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  gelu_fwd_kernel<<<grid_for(n, 256), 256, 0, s>>>(f, n, reinterpret_cast<__nv_bfloat16*>(out16), out32);
  PLLB_LAUNCH_CHECK("gelu_fwd_kernel");
  return PLLB_OK;
}

int launch_train_gelu_bwd(float* dg, const float* f, int64_t n, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  gelu_bwd_kernel<<<grid_for(n, 256), 256, 0, s>>>(dg, f, n);
  PLLB_LAUNCH_CHECK("gelu_bwd_kernel");
  return PLLB_OK;
}

int launch_train_cast_transpose(const void* src, bool src_bf16, int R, int C, int Rp, void* dst16, void* dstT,
                                cudaStream_t s) {
  if (C <= 0 || Rp <= 0) return PLLB_OK;
  dim3 grid((unsigned)ceil_div(C, 32), (unsigned)ceil_div(Rp, 32));
  if (src_bf16)
    cast_transpose_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(src), R, C, Rp,
                                                             reinterpret_cast<__nv_bfloat16*>(dst16),
                                                             reinterpret_cast<__nv_bfloat16*>(dstT));
  else
    cast_transpose_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(src), R, C, Rp,
                                                     reinterpret_cast<__nv_bfloat16*>(dst16),
                                                     reinterpret_cast<__nv_bfloat16*>(dstT));
  PLLB_LAUNCH_CHECK("cast_transpose_kernel");
  return PLLB_OK;
}

int launch_train_attn_fwd(const void* qkv, const int32_t* n_valid, int R, int T, int H, int NH, TrainDrop drop, uint32_t site,
                          void* ctx, float* lse, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const size_t smem = sizeof(float) * RW * (64 + (size_t)T);
  attn_fwd_train_kernel<<<(int)ceil_div((int64_t)R * NH, RW), RW * 32, smem, s>>>(
      reinterpret_cast<const __nv_bfloat16*>(qkv), n_valid, R, T, H, NH, drop, site, reinterpret_cast<__nv_bfloat16*>(ctx), lse);
  PLLB_LAUNCH_CHECK("attn_fwd_train_kernel");
  return PLLB_OK;
}

int launch_train_attn_bwd(const void* qkv, const float* dctx, const float* lse, const int32_t* n_valid, int R, int T, int H,
                          int NH, TrainDrop drop, uint32_t site, float* dqkv, float* Dscratch, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const size_t smem = sizeof(float) * RW * (128 + 2 * (size_t)T);
  const int grid = (int)ceil_div((int64_t)R * NH, RW);
  attn_bwd_q_kernel<<<grid, RW * 32, smem, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), dctx, lse, n_valid, R, T, H, NH,
                                                drop, site, dqkv, Dscratch);
  PLLB_LAUNCH_CHECK("attn_bwd_q_kernel");
  attn_bwd_kv_kernel<<<grid, RW * 32, smem, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv), dctx, lse, Dscratch, n_valid, R,
                                                 T, H, NH, drop, site, dqkv);
  PLLB_LAUNCH_CHECK("attn_bwd_kv_kernel");
  return PLLB_OK;
}

int launch_train_ce(const float* logits, const int32_t* labels, int R, int V, int Vp, float* loss_rows, void* dlogits,
                    float* out_loss, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  ce_kernel<<<R, 256, 0, s>>>(logits, labels, V, Vp, loss_rows, reinterpret_cast<__nv_bfloat16*>(dlogits));
  PLLB_LAUNCH_CHECK("ce_kernel");
  loss_mean_kernel<<<1, 256, 0, s>>>(loss_rows, R, out_loss);
  PLLB_LAUNCH_CHECK("loss_mean_kernel");
  return PLLB_OK;
}

int launch_train_scale(float* x, int64_t n, float alpha, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  scale_kernel<<<grid_for(n, 256), 256, 0, s>>>(x, n, alpha);
  PLLB_LAUNCH_CHECK("scale_kernel");
  return PLLB_OK;
}

int launch_train_embed_bwd(const float* dz, const int32_t* ids, int B, int T, int H, int max_pos, int pad_id, float* dword,
                           float* dpos, float* dtype0, float* scratch, cudaStream_t s) {
  const int R = B * T;
  if (R <= 0) return PLLB_OK;
  pos_grad_kernel<<<grid_for((int64_t)max_pos * H, 256), 256, 0, s>>>(dz, B, T, H, max_pos, dpos);
  PLLB_LAUNCH_CHECK("pos_grad_kernel");
  int rc = launch_train_colsum(dz, false, nullptr, R, H, dtype0, nullptr, scratch, s);
  if (rc) return rc;
  word_grad_kernel<<<R, 256, 0, s>>>(dz, ids, R, H, pad_id, dword);
  PLLB_LAUNCH_CHECK("word_grad_kernel");
  return PLLB_OK;
}

int launch_train_adamw(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                       float wd, const TrainStepParams* scalars, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  adamw_kernel<<<grid_for(n, 256), 256, 0, s>>>(p, g, m, v, n, lr, beta1, beta2, eps, wd, scalars);
  PLLB_LAUNCH_CHECK("adamw_kernel");
  return PLLB_OK;
}

int launch_train_cls_fwd(const float* h, const float* w, const float* b, int B, int T, int H, float* scores, cudaStream_t s) {
  if (B <= 0) return PLLB_OK;
  const int grid = (int)ceil_div(B, RW);
  DISPATCH_NV(H, cls_fwd_kernel<NV><<<grid, RW * 32, 0, s>>>(h, w, b, B, T, scores));
  PLLB_LAUNCH_CHECK("cls_fwd_kernel");
  return PLLB_OK;
}

int launch_train_cls_loss(const float* scores, const float* target, const float* am, const float* err, const int32_t* group,
                          int B, float md_weight, float mwer_weight, float am_weight, float* dscore, float* out_loss,
                          cudaStream_t s) {
  if (B <= 0) return PLLB_OK;
  cls_loss_kernel<<<1, 256, 0, s>>>(scores, target, am, err, group, B, md_weight, mwer_weight, am_weight, dscore, out_loss);
  PLLB_LAUNCH_CHECK("cls_loss_kernel");
  return PLLB_OK;
}

int launch_train_cls_bwd(const float* h, const float* w, const float* dscore, int B, int T, int H, float* dw, float* db,
                         float* dh, cudaStream_t s) {
  if (B <= 0) return PLLB_OK;
  cls_bwd_kernel<<<1 + grid_for((int64_t)B * T * H, 256), 256, 0, s>>>(h, w, dscore, B, T, H, dw, db, dh);
  PLLB_LAUNCH_CHECK("cls_bwd_kernel");
  return PLLB_OK;
}

// ================================================================== BART fine-tuning (pllb_s2s_train_*)
namespace {

// out = [dropout](LN(shared[id] * scale + pos[r % T]))   (BART embeddings; pos already points at row 2 of the table)
template <int NV>
__global__ void __launch_bounds__(RW * 32)
bart_embed_kernel(const int32_t* __restrict__ ids, int T, const float* __restrict__ word, float scale,
                  const float* __restrict__ pos, const float* __restrict__ g, const float* __restrict__ b, float eps, int R,
                  TrainDrop drop, uint32_t site, float* __restrict__ out32, __nv_bfloat16* __restrict__ out16,
                  float* __restrict__ xhat, float* __restrict__ rstd) {
  constexpr int H = NV * 32;
  const int r = blockIdx.x * RW + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (r >= R) return;
  const int id = ids[r], p = r % T;
  float v[NV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    v[i] = word[(size_t)id * H + c] * scale + pos[(size_t)p * H + c];
    s += v[i];
  }
  const float mean = wsum(s) * (1.f / H);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) { const float d = v[i] - mean; q += d * d; }
  const float rs = rsqrtf(wsum(q) * (1.f / H) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int c = lane + 32 * i;
    const size_t e = (size_t)r * H + c;
    const float xh = (v[i] - mean) * rs;
    const float o = (xh * g[c] + b[c]) * drop_factor(drop, site, e);
    xhat[e] = xh;
    out32[e] = o;
    out16[e] = __float2bfloat16_rn(o);
  }
  if (lane == 0) rstd[r] = rs;
}

// Attention of B sequences whose Tq query rows (q, row stride ldq) attend to Tk key / value rows of the same
// sequence (k, v, row stride ldkv), warp per (query row, head).  CAUSAL: Tq == Tk and query i sees keys <= i
// (the decoder's self-attention); otherwise the keys < n_valid[seq] (cross-attention over the encoder rows).
__device__ __forceinline__ int s2s_key_limit(bool causal, int i, const int32_t* n_valid, int seq) {
  return causal ? i + 1 : n_valid[seq];
}

template <bool CAUSAL>
__global__ void __launch_bounds__(RW * 32, 8)     // without the occupancy hint ptxas spills 4 bytes in the cross form
attn_fwd_s2s_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                    const __nv_bfloat16* __restrict__ v, int ldq, int ldkv, const int32_t* __restrict__ n_valid, int Rq,
                    int Tq, int Tk, int NH, TrainDrop drop, uint32_t site, __nv_bfloat16* __restrict__ ctx,
                    float* __restrict__ lse_out) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= Rq * NH) return;
  const int r = item / NH, h = item % NH, seq = r / Tq, i = r % Tq, H = NH * 64;
  const int nk = s2s_key_limit(CAUSAL, i, n_valid, seq);
  float* sq = smem + (size_t)w * (64 + Tk);
  float* sp = sq + 64;
  const __nv_bfloat16* kb = k + (size_t)seq * Tk * ldkv + h * 64;
  const __nv_bfloat16* vb = v + (size_t)seq * Tk * ldkv + h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(q + (size_t)r * ldq + h * 64 + 2 * lane));
    sq[2 * lane] = f.x; sq[2 * lane + 1] = f.y;
  }
  __syncwarp();
  float m = -INFINITY;
  for (int j = lane; j < nk; j += 32) {
    const float s = dot64_bf16(sq, kb + (size_t)j * ldkv) * 0.125f;
    sp[j] = s;
    m = fmaxf(m, s);
  }
  m = wmax(m);
  float l = 0.f;
  for (int j = lane; j < nk; j += 32) l += __expf(sp[j] - m);
  const float lse = m + __logf(wsum(l));
  const uint64_t pbase = ((uint64_t)(seq * NH + h) * Tq + i) * Tk;
  for (int j = lane; j < nk; j += 32) sp[j] = __expf(sp[j] - lse) * drop_factor(drop, site, pbase + j);
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
  for (int j = 0; j < nk; ++j) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(vb + (size_t)j * ldkv + 2 * lane));
    a0 += sp[j] * f.x; a1 += sp[j] * f.y;
  }
  *reinterpret_cast<__nv_bfloat162*>(ctx + (size_t)r * H + h * 64 + 2 * lane) = __floats2bfloat162_rn(a0, a1);
  if (lane == 0) lse_out[item] = lse;
}

// dq of query row r (fp32, row stride lddq) and D_r = sum_j P_rj dP_rj for the dk / dv pass
template <bool CAUSAL>
__global__ void __launch_bounds__(RW * 32)
attn_bwd_q_s2s_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                      const __nv_bfloat16* __restrict__ v, int ldq, int ldkv, const float* __restrict__ dctx,
                      const float* __restrict__ lse, const int32_t* __restrict__ n_valid, int Rq, int Tq, int Tk, int NH,
                      TrainDrop drop, uint32_t site, float* __restrict__ dq, int lddq, float* __restrict__ Dout) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= Rq * NH) return;
  const int r = item / NH, h = item % NH, seq = r / Tq, i = r % Tq, H = NH * 64;
  const int nk = s2s_key_limit(CAUSAL, i, n_valid, seq);
  float* sq = smem + (size_t)w * (128 + 2 * Tk);
  float* sdo = sq + 64;
  float* sp = sdo + 64;
  float* sds = sp + Tk;
  const __nv_bfloat16* kb = k + (size_t)seq * Tk * ldkv + h * 64;
  const __nv_bfloat16* vb = v + (size_t)seq * Tk * ldkv + h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(q + (size_t)r * ldq + h * 64 + 2 * lane));
    sq[2 * lane] = f.x; sq[2 * lane + 1] = f.y;
    const float2 g = *reinterpret_cast<const float2*>(dctx + (size_t)r * H + h * 64 + 2 * lane);
    sdo[2 * lane] = g.x; sdo[2 * lane + 1] = g.y;
  }
  __syncwarp();
  const float ls = lse[item];
  const uint64_t pbase = ((uint64_t)(seq * NH + h) * Tq + i) * Tk;
  float dpart = 0.f;
  for (int j = lane; j < nk; j += 32) {
    const float p = __expf(dot64_bf16(sq, kb + (size_t)j * ldkv) * 0.125f - ls);
    const float dp = dot64_bf16(sdo, vb + (size_t)j * ldkv) * drop_factor(drop, site, pbase + j);
    sp[j] = p; sds[j] = dp;
    dpart += p * dp;
  }
  const float D = wsum(dpart);
  for (int j = lane; j < nk; j += 32) sds[j] = sp[j] * (sds[j] - D);
  __syncwarp();
  float a0 = 0.f, a1 = 0.f;
#pragma unroll 4
  for (int j = 0; j < nk; ++j) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(kb + (size_t)j * ldkv + 2 * lane));
    a0 += sds[j] * f.x; a1 += sds[j] * f.y;
  }
  *reinterpret_cast<float2*>(dq + (size_t)r * lddq + h * 64 + 2 * lane) = make_float2(a0 * 0.125f, a1 * 0.125f);
  if (lane == 0) Dout[item] = D;
}

// dk and dv of key row rk (fp32, row stride lddkv): sums over the queries that see it, in query order (CAUSAL: i >= j;
// cross: all Tq decoder rows of the sentence).  A masked key gets zero.
template <bool CAUSAL>
__global__ void __launch_bounds__(RW * 32)
attn_bwd_kv_s2s_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ k,
                       const __nv_bfloat16* __restrict__ v, int ldq, int ldkv, const float* __restrict__ dctx,
                       const float* __restrict__ lse, const float* __restrict__ Dq, const int32_t* __restrict__ n_valid,
                       int Rk, int Tq, int Tk, int NH, TrainDrop drop, uint32_t site, float* __restrict__ dk,
                       float* __restrict__ dv, int lddkv) {
  extern __shared__ float smem[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int item = blockIdx.x * RW + w;
  if (item >= Rk * NH) return;
  const int rk = item / NH, h = item % NH, seq = rk / Tk, j = rk % Tk, H = NH * 64;
  float2* dk_out = reinterpret_cast<float2*>(dk + (size_t)rk * lddkv + h * 64 + 2 * lane);
  float2* dv_out = reinterpret_cast<float2*>(dv + (size_t)rk * lddkv + h * 64 + 2 * lane);
  if (!CAUSAL && j >= n_valid[seq]) {
    *dk_out = make_float2(0.f, 0.f);
    *dv_out = make_float2(0.f, 0.f);
    return;
  }
  const int i0 = CAUSAL ? j : 0;
  float* sk = smem + (size_t)w * (128 + 2 * Tq);
  float* sv = sk + 64;
  float* sds = sv + 64;
  float* spd = sds + Tq;
  const __nv_bfloat16* qb = q + (size_t)seq * Tq * ldq + h * 64;
  {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(k + (size_t)rk * ldkv + h * 64 + 2 * lane));
    sk[2 * lane] = f.x; sk[2 * lane + 1] = f.y;
    const float2 g = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(v + (size_t)rk * ldkv + h * 64 + 2 * lane));
    sv[2 * lane] = g.x; sv[2 * lane + 1] = g.y;
  }
  __syncwarp();
  for (int i = i0 + lane; i < Tq; i += 32) {
    const int ri = seq * Tq + i;
    const float p = __expf(dot64_bf16(sk, qb + (size_t)i * ldq) * 0.125f - lse[(size_t)ri * NH + h]);
    const float sc = drop_factor(drop, site, ((uint64_t)(seq * NH + h) * Tq + i) * Tk + j);
    const float dp = dot64_f32(sv, dctx + (size_t)ri * H + h * 64) * sc;
    sds[i] = p * (dp - Dq[(size_t)ri * NH + h]);
    spd[i] = p * sc;
  }
  __syncwarp();
  float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
#pragma unroll 4
  for (int i = i0; i < Tq; ++i) {
    const int ri = seq * Tq + i;
    const float2 qq = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(qb + (size_t)i * ldq + 2 * lane));
    const float2 g = *reinterpret_cast<const float2*>(dctx + (size_t)ri * H + h * 64 + 2 * lane);
    k0 += sds[i] * qq.x; k1 += sds[i] * qq.y;
    v0 += spd[i] * g.x; v1 += spd[i] * g.y;
  }
  *dk_out = make_float2(k0 * 0.125f, k1 * 0.125f);
  *dv_out = make_float2(v0, v1);
}

// Cross entropy with ignore_index -100: as ce_kernel on a row whose label is in [0, V); an ignored row has loss 0
// and a zero dlogits row (bf16, unscaled: the 1/N of the mean is applied in fp32 by the consumers).
__global__ void __launch_bounds__(256)
ce_ignore_kernel(const float* __restrict__ logits, const int32_t* __restrict__ labels, int V, int Vp,
                 float* __restrict__ loss_rows, __nv_bfloat16* __restrict__ dlogits) {
  __shared__ float red[8];
  __shared__ float bc;
  const int r = blockIdx.x, tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int label = labels[r];
  if (label < 0) {
    if (tid == 0) loss_rows[r] = 0.f;
    if (dlogits)
      for (int c = tid; c < Vp; c += 256) dlogits[(size_t)r * Vp + c] = __float2bfloat16_rn(0.f);
    return;
  }
  const float* x = logits + (size_t)r * Vp;
  float m = -INFINITY;
  for (int c = tid; c < V; c += 256) m = fmaxf(m, x[c]);
  m = wmax(m);
  if (lane == 0) red[w] = m;
  __syncthreads();
  if (tid == 0) { float t = red[0]; for (int k = 1; k < 8; ++k) t = fmaxf(t, red[k]); bc = t; }
  __syncthreads();
  m = bc;
  float s = 0.f;
  for (int c = tid; c < V; c += 256) s += __expf(x[c] - m);
  s = wsum(s);
  __syncthreads();
  if (lane == 0) red[w] = s;
  __syncthreads();
  if (tid == 0) { float t = 0.f; for (int k = 0; k < 8; ++k) t += red[k]; bc = m + logf(t); }
  __syncthreads();
  const float lse = bc;
  if (tid == 0) loss_rows[r] = lse - x[label];
  if (dlogits) {
    __nv_bfloat16* d = dlogits + (size_t)r * Vp;
    for (int c = tid; c < Vp; c += 256) {
      float g = 0.f;
      if (c < V) g = __expf(x[c] - lse) - (c == label ? 1.f : 0.f);
      d[c] = __float2bfloat16_rn(g);
    }
  }
}

// out[0] = the mean of the per-row losses over the N rows with a label (fixed order, double accumulation);
// out[1] = 1 / N in fp32, the factor the backward pass applies.  Single block; N >= 1 is checked on the host.
__global__ void __launch_bounds__(256)
loss_mean_valid_kernel(const float* __restrict__ loss_rows, const int32_t* __restrict__ labels, int R, float* __restrict__ out) {
  __shared__ double red[256];
  __shared__ int cnt[256];
  double a = 0.0;
  int n = 0;
  for (int r = threadIdx.x; r < R; r += 256)
    if (labels[r] >= 0) { a += (double)loss_rows[r]; ++n; }
  red[threadIdx.x] = a;
  cnt[threadIdx.x] = n;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { red[threadIdx.x] += red[threadIdx.x + o]; cnt[threadIdx.x] += cnt[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    out[0] = (float)(red[0] / (double)cnt[0]);
    out[1] = 1.f / (float)cnt[0];
  }
}

// x *= alpha[0], alpha read from device memory (the 1 / N of a batch inside a captured graph)
__global__ void scale_dev_kernel(float* __restrict__ x, int64_t n, const float* __restrict__ alpha) {
  const float a = *alpha;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) x[i] *= a;
}

}  // namespace

int launch_train_bart_embed(const int32_t* ids, int T, const float* word, float scale, const float* pos, const float* g,
                            const float* b, float eps, int R, int H, TrainDrop drop, uint32_t site, float* out32, void* out16,
                            float* xhat, float* rstd, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  const int grid = (int)ceil_div(R, RW);
  DISPATCH_NV(H, bart_embed_kernel<NV><<<grid, RW * 32, 0, s>>>(ids, T, word, scale, pos, g, b, eps, R, drop, site, out32,
                                                               reinterpret_cast<__nv_bfloat16*>(out16), xhat, rstd));
  PLLB_LAUNCH_CHECK("bart_embed_kernel");
  return PLLB_OK;
}

int launch_train_bart_embed_bwd(float* dz, const int32_t* ids, int B, int T, int H, int pos_rows, int pad_id, float scale,
                                float* dword, float* dpos, cudaStream_t s) {
  const int R = B * T;
  if (R <= 0) return PLLB_OK;
  pos_grad_kernel<<<grid_for((int64_t)pos_rows * H, 256), 256, 0, s>>>(dz, B, T, H, pos_rows, dpos);
  PLLB_LAUNCH_CHECK("pos_grad_kernel");
  if (scale != 1.f) {           // the lookup is shared[id] * scale: each occurrence sends dz * scale
    scale_kernel<<<grid_for((int64_t)R * H, 256), 256, 0, s>>>(dz, (int64_t)R * H, scale);
    PLLB_LAUNCH_CHECK("scale_kernel");
  }
  word_grad_kernel<<<R, 256, 0, s>>>(dz, ids, R, H, pad_id, dword);
  PLLB_LAUNCH_CHECK("word_grad_kernel");
  return PLLB_OK;
}

int launch_train_attn_s2s_fwd(const S2sAttn& a, TrainDrop drop, uint32_t site, void* ctx, float* lse, cudaStream_t s) {
  const int Rq = a.B * a.Tq;
  if (Rq <= 0) return PLLB_OK;
  const size_t smem = sizeof(float) * RW * (64 + (size_t)a.Tk);
  const int grid = (int)ceil_div((int64_t)Rq * a.NH, RW);
  const auto* q = reinterpret_cast<const __nv_bfloat16*>(a.q);
  const auto* k = reinterpret_cast<const __nv_bfloat16*>(a.k);
  const auto* v = reinterpret_cast<const __nv_bfloat16*>(a.v);
  auto* c16 = reinterpret_cast<__nv_bfloat16*>(ctx);
  if (a.causal)
    attn_fwd_s2s_kernel<true><<<grid, RW * 32, smem, s>>>(q, k, v, a.ldq, a.ldkv, a.n_valid, Rq, a.Tq, a.Tk, a.NH, drop, site, c16, lse);
  else
    attn_fwd_s2s_kernel<false><<<grid, RW * 32, smem, s>>>(q, k, v, a.ldq, a.ldkv, a.n_valid, Rq, a.Tq, a.Tk, a.NH, drop, site, c16, lse);
  PLLB_LAUNCH_CHECK("attn_fwd_s2s_kernel");
  return PLLB_OK;
}

int launch_train_attn_s2s_bwd(const S2sAttn& a, const float* dctx, const float* lse, TrainDrop drop, uint32_t site, float* dq,
                              int lddq, float* dk, float* dv, int lddkv, float* Dscratch, cudaStream_t s) {
  const int Rq = a.B * a.Tq, Rk = a.B * a.Tk;
  if (Rq <= 0) return PLLB_OK;
  const auto* q = reinterpret_cast<const __nv_bfloat16*>(a.q);
  const auto* k = reinterpret_cast<const __nv_bfloat16*>(a.k);
  const auto* v = reinterpret_cast<const __nv_bfloat16*>(a.v);
  const size_t smem_q = sizeof(float) * RW * (128 + 2 * (size_t)a.Tk), smem_kv = sizeof(float) * RW * (128 + 2 * (size_t)a.Tq);
  const int grid_q = (int)ceil_div((int64_t)Rq * a.NH, RW), grid_kv = (int)ceil_div((int64_t)Rk * a.NH, RW);
  if (a.causal)
    attn_bwd_q_s2s_kernel<true><<<grid_q, RW * 32, smem_q, s>>>(q, k, v, a.ldq, a.ldkv, dctx, lse, a.n_valid, Rq, a.Tq, a.Tk,
                                                               a.NH, drop, site, dq, lddq, Dscratch);
  else
    attn_bwd_q_s2s_kernel<false><<<grid_q, RW * 32, smem_q, s>>>(q, k, v, a.ldq, a.ldkv, dctx, lse, a.n_valid, Rq, a.Tq, a.Tk,
                                                                a.NH, drop, site, dq, lddq, Dscratch);
  PLLB_LAUNCH_CHECK("attn_bwd_q_s2s_kernel");
  if (a.causal)
    attn_bwd_kv_s2s_kernel<true><<<grid_kv, RW * 32, smem_kv, s>>>(q, k, v, a.ldq, a.ldkv, dctx, lse, Dscratch, a.n_valid, Rk,
                                                                  a.Tq, a.Tk, a.NH, drop, site, dk, dv, lddkv);
  else
    attn_bwd_kv_s2s_kernel<false><<<grid_kv, RW * 32, smem_kv, s>>>(q, k, v, a.ldq, a.ldkv, dctx, lse, Dscratch, a.n_valid, Rk,
                                                                   a.Tq, a.Tk, a.NH, drop, site, dk, dv, lddkv);
  PLLB_LAUNCH_CHECK("attn_bwd_kv_s2s_kernel");
  return PLLB_OK;
}

int launch_train_ce_ignore(const float* logits, const int32_t* labels, int R, int V, int Vp, float* loss_rows, void* dlogits,
                           float* out_loss2, cudaStream_t s) {
  if (R <= 0) return PLLB_OK;
  ce_ignore_kernel<<<R, 256, 0, s>>>(logits, labels, V, Vp, loss_rows, reinterpret_cast<__nv_bfloat16*>(dlogits));
  PLLB_LAUNCH_CHECK("ce_ignore_kernel");
  loss_mean_valid_kernel<<<1, 256, 0, s>>>(loss_rows, labels, R, out_loss2);
  PLLB_LAUNCH_CHECK("loss_mean_valid_kernel");
  return PLLB_OK;
}

int launch_train_scale_dev(float* x, int64_t n, const float* alpha, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  scale_dev_kernel<<<grid_for(n, 256), 256, 0, s>>>(x, n, alpha);
  PLLB_LAUNCH_CHECK("scale_dev_kernel");
  return PLLB_OK;
}

}  // namespace pllb
