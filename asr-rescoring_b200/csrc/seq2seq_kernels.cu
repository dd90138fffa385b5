// seq2seq_kernels.cu — the small kernels of greedy encoder-decoder generation (pllb_generate).
//
// A decoder step over the rows in flight is: embedding + LayerNorm, then per layer the QKV GEMM,
// single-query self-attention over the row's KV cache, attention-output GEMM + LayerNorm, cross-Q
// GEMM, single-query cross-attention over the row's encoder K/V, output GEMM + LayerNorm and the
// FFN; then the LM head GEMM with the EPI_ARGMAX epilogue and argmax_finish.  The GEMMs are the
// tcgen05 kernels of gemm_tcgen05.cu / gemm_ln_tcgen05.cu; this file holds everything else.
// Beam search (pllb_generate_beam) adds beam_select_kernel, which merges the EPI_TOPK8 / EPI_TOPK16
// partials and carries the beam bookkeeping, and a slot-table form of the self-attention.
// fp32 arithmetic, no atomics except the integer counts of finished rows / frozen sentences: a run is
// bit-deterministic.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>

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
// SLOT (beam search, self form): key j < self_t of row r is cache row slot[r * max_len + j] instead of
// r * max_len + j, so beams that share a prefix share its cache rows; the trailing `slot` parameter is
// unused otherwise.
template <bool FP16, bool SLOT>
__global__ void __launch_bounds__(128, 4) decode_attention_kernel(
    const uint16_t* __restrict__ q, int q_stride, const uint16_t* kv, int64_t kv_stride,
    const int32_t* __restrict__ key_start, const int32_t* __restrict__ key_len, int self_t, int max_len,
    const uint16_t* __restrict__ new_kv, int new_kv_stride, uint16_t* kv_cache, uint16_t* __restrict__ ctx, int rows,
    int H, int NH, int max_keys, const int32_t* __restrict__ slot) {
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
  // SLOT: cache row of key j (keys before self_t through the slot table, key self_t the row's own)
  auto key_row = [&](int j) -> const uint16_t* {
    const int64_t cr = j < self_t ? (int64_t)slot[(size_t)r * max_len + j] : (int64_t)r * max_len + self_t;
    return kv_cache + (size_t)cr * (size_t)(2 * H);
  };
  float m = -INFINITY;
  for (int j = lane; j < n; j += 32) {
    const uint16_t* krow;
    if constexpr (SLOT) krow = key_row(j) + h * 64;
    else krow = base + (size_t)j * stride + h * 64;
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
    uint32_t u;
    if constexpr (SLOT) u = *reinterpret_cast<const uint32_t*>(key_row(j) + H + h * 64 + 2 * lane);
    else u = *reinterpret_cast<const uint32_t*>(vcol + (size_t)j * stride);
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

// ---------------------------------------------------------------------------------------- beam search
// DESIGN.md §3.12.  (value, index) orders of the selection: higher value first, then lower index.
__device__ __forceinline__ bool beats(float v, int i, float w, int j) { return v > w || (v == w && i < j); }

__device__ __forceinline__ void lse_merge(float& m, float& s, float m2, float s2) {
  if (m2 == -INFINITY) return;
  if (m == -INFINITY) { m = m2; s = s2; return; }
  const float nm = fmaxf(m, m2);
  s = s * expf(m - nm) + s2 * expf(m2 - nm);
  m = nm;
}

__global__ void beam_init_kernel(BeamState st) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r == 0) *st.frozen_count = 0;
  if (r < st.n) st.sent_flags[r] = 0;
  if (r >= st.n * st.K) return;
  st.ids_cur[(size_t)r * st.max_len] = st.start_id;
  st.ids_next[(size_t)r * st.max_len] = st.start_id;
  int32_t* f = st.fin_ids + (size_t)r * st.max_len;
  f[0] = st.start_id;
  for (int j = 1; j < st.max_len; ++j) f[j] = st.pad_id;
  st.fin_len[r] = 1;
  st.fin_score[r] = -1e9f;
  st.fin_flag[r] = 0;
  st.run_score[r] = r % st.K == 0 ? 0.f : -1e9f;
  st.parent[r] = r;
}

// One CTA of 256 threads per sentence; warp b < K merges beam row b's partials, warp 0 then selects the
// sentence's top 2K candidates and thread 0 applies items 3-7 of the contract in fp32, in a fixed order.
// Dynamic shared memory: K * max_len ints (the old finished ids while the slots are rewritten).
template <int KS>
__global__ void __launch_bounds__(256) beam_select_kernel(const float2* __restrict__ parts, int n_parts, int vocab,
                                                          BeamState st, int t) {
  extern __shared__ int32_t stage[];
  __shared__ float c_val[8][KS];
  __shared__ int c_tok[8][KS];
  __shared__ float s_val[16];
  __shared__ int s_tok[16], s_beam[16];
  __shared__ int n_par[8], n_tok[8], f_src[8], f_flag[8];
  __shared__ float n_rs[8], f_score[8];
  __shared__ int s_frozen, s_changed;
  const int i = blockIdx.x;
  const int K = st.K, TK = 2 * K, ML = st.max_len, rows = st.n * st.K;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row0 = i * K;
  if (threadIdx.x == 0) { s_frozen = (st.sent_flags[i] & 2) != 0; s_changed = 0; }
  __syncthreads();
  const bool frozen = s_frozen != 0;
  const int forced = t == ML - 1 && st.forced_eos >= 0 ? st.forced_eos : t == 1 && st.forced_bos >= 0 ? st.forced_bos : -1;
  if (!frozen && warp < K) {
    const int r = row0 + warp;
    const float rs = st.run_score[r];
    if (forced >= 0) {
      // log-probabilities 0 at the forced id and -inf elsewhere: the -inf ones in column order
      if (lane < TK) {
        c_val[warp][lane] = lane == 0 ? 0.f + rs : -INFINITY;
        c_tok[warp][lane] = lane == 0 ? forced : lane - 1 < forced ? lane - 1 : lane;
      }
    } else {
      const float2* lp = parts + (size_t)r * n_parts;
      float m = -INFINITY, sum = 0.f;
      for (int q = lane; q < n_parts; q += 32) {
        const float2 v = lp[q];
        lse_merge(m, sum, v.x, v.y);
      }
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, sum, o);
        // both lanes of a pair merge the same two values in the same order
        float a = m, b = sum, c = m2, d = s2;
        if ((lane & o) != 0) { a = m2; b = s2; c = m; d = sum; }
        lse_merge(a, b, c, d);
        m = a;
        sum = b;
      }
      const float logs = logf(sum);
      float tv[KS];
      int tc[KS];
#pragma unroll
      for (int k = 0; k < KS; ++k) { tv[k] = -INFINITY; tc[k] = INT_MAX; }
      const float2* tp = parts + (size_t)rows * n_parts + (size_t)r * n_parts * KS;
      for (int q = lane; q < n_parts; q += 32) {
        for (int e = 0; e < KS; ++e) {            // each list descends: stop at the first entry that stays out
          const float2 v = tp[(size_t)q * KS + e];
          const int col = __float_as_int(v.y);
          if (!beats(v.x, col, tv[KS - 1], tc[KS - 1])) break;
          tv[KS - 1] = v.x;
          tc[KS - 1] = col;
#pragma unroll
          for (int k = KS - 1; k > 0; --k)
            if (beats(tv[k], tc[k], tv[k - 1], tc[k - 1])) {
              const float fv = tv[k]; tv[k] = tv[k - 1]; tv[k - 1] = fv;
              const int fc = tc[k]; tc[k] = tc[k - 1]; tc[k - 1] = fc;
            }
        }
      }
      for (int k = 0; k < TK; ++k) {              // warp merge of the lanes' sorted lists
        float bv = tv[0];
        int bc = tc[0], bl = lane;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
          const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
          const int oc = __shfl_xor_sync(0xffffffffu, bc, o), ol = __shfl_xor_sync(0xffffffffu, bl, o);
          if (beats(ov, oc, bv, bc) || (ov == bv && oc == bc && ol < bl)) { bv = ov; bc = oc; bl = ol; }
        }
        if (lane == bl) {
#pragma unroll
          for (int q = 0; q < KS - 1; ++q) { tv[q] = tv[q + 1]; tc[q] = tc[q + 1]; }
          tv[KS - 1] = -INFINITY;
          tc[KS - 1] = INT_MAX;
        }
        if (lane == 0) {
          c_val[warp][k] = ((bv - m) - logs) + rs;   // log_softmax as (x - max) - log(sum), plus the beam score
          c_tok[warp][k] = min(bc, vocab - 1);
        }
      }
    }
  }
  __syncthreads();
  if (!frozen && warp == 0) {
    // the sentence's top 2K of the K * 2K candidates, flat index beam * vocab + token on ties
    float v[4];
    int fl[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int e = lane + 32 * q;
      const bool ok = e < K * TK;
      v[q] = ok ? c_val[e / TK][e % TK] : -INFINITY;
      fl[q] = ok ? (e / TK) * vocab + c_tok[e / TK][e % TK] : INT_MAX;
    }
    for (int k = 0; k < TK; ++k) {
      float bv = -INFINITY;
      int bf = INT_MAX, bq = -1;
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (fl[q] != INT_MAX && (bq < 0 || beats(v[q], fl[q], bv, bf))) { bv = v[q]; bf = fl[q]; bq = q; }
      int bl = bq >= 0 ? lane : 32;
#pragma unroll
      for (int o = 16; o; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int of = __shfl_xor_sync(0xffffffffu, bf, o), ol = __shfl_xor_sync(0xffffffffu, bl, o);
        if (ol < 32 && (bl == 32 || beats(ov, of, bv, bf))) { bv = ov; bf = of; bl = ol; }
      }
      if (lane == bl) fl[bq] = INT_MAX;             // used
      if (lane == 0) {
        s_val[k] = bv;
        s_beam[k] = bf / vocab;
        s_tok[k] = bf % vocab;
      }
    }
    __syncwarp();
    if (lane == 0) {
      const bool last = t == ML - 1;
      bool hit[16];
      float pen[16];
      for (int c = 0; c < TK; ++c) {
        hit[c] = s_tok[c] == st.eos_id || last;
        pen[c] = hit[c] ? s_val[c] + -1e9f : s_val[c];
      }
      // running beams: top K of the penalised candidates
      bool used[24];
      for (int c = 0; c < 24; ++c) used[c] = false;
      for (int k = 0; k < K; ++k) {
        int b = -1;
        for (int c = 0; c < TK; ++c)
          if (!used[c] && (b < 0 || beats(pen[c], c, pen[b], b))) b = c;
        used[b] = true;
        n_par[k] = row0 + s_beam[b];
        n_tok[k] = s_tok[b];
        n_rs[k] = pen[b];
      }
      // finished slots: top K of the old slots followed by the 2K normalised candidates
      float fs[24];
      bool ff[24];
      bool all_fin = true;
      for (int j = 0; j < K; ++j) {
        fs[j] = st.fin_score[row0 + j];
        ff[j] = st.fin_flag[row0 + j] != 0;
        all_fin = all_fin && ff[j];
      }
      const int flags = st.sent_flags[i];
      const bool unsat = (flags & 1) == 0;
      const float norm = (float)pow((double)t, (double)st.length_penalty);
      for (int c = 0; c < TK; ++c) {
        float sc = s_val[c] / norm;
        if (all_fin && st.early_stopping == 1) sc += -1e9f;
        if (!unsat) sc += -1e9f;
        const bool jf = c < K && hit[c];
        if (!jf) sc += -1e9f;
        fs[K + c] = sc;
        ff[K + c] = jf;
      }
      for (int c = 0; c < 24; ++c) used[c] = false;
      bool changed = false;
      for (int k = 0; k < K; ++k) {
        int b = -1;
        for (int c = 0; c < K + TK; ++c)
          if (!used[c] && (b < 0 || beats(fs[c], c, fs[b], b))) b = c;
        used[b] = true;
        f_src[k] = b;
        f_score[k] = fs[b];
        f_flag[k] = ff[b];
        changed = changed || b != k;
      }
      // early-stop heuristic with t' = t + 1, then freezing
      const double Lh = st.early_stopping == 2 && st.length_penalty > 0.f ? (double)(ML - 1) : (double)t;
      const float best = n_rs[0] / (float)pow(Lh, (double)st.length_penalty);
      float mn = f_score[0];
      bool all_new = true;
      for (int k = 0; k < K; ++k) { mn = fminf(mn, f_score[k]); all_new = all_new && f_flag[k]; }
      bool any = false;
      for (int k = 0; k < K; ++k) any = any || best > (f_flag[k] ? mn : -1e9f);
      const bool unsat_new = unsat && any;
      const bool frz = !unsat_new || (st.early_stopping == 1 && all_new);
      st.sent_flags[i] = (unsat_new ? 0 : 1) | (frz ? 2 : 0);
      if (frz) atomicAdd(st.frozen_count, 1);
      s_changed = changed;
    }
  }
  __syncthreads();
  // a frozen sentence keeps its rows: each is its own parent and feeds pad_id from here on
  for (int k = warp; k < K; k += 8) {
    const int r = row0 + k;
    const int par = frozen ? r : n_par[k];
    const int tok = frozen ? st.pad_id : n_tok[k];
    for (int j = lane; j <= t; j += 32) {
      st.ids_next[(size_t)r * ML + j] = j < t ? st.ids_cur[(size_t)par * ML + j] : tok;
      if (j < t) st.slot_next[(size_t)r * ML + j] = j < t - 1 ? st.slot_cur[(size_t)par * ML + j] : par * ML + t - 1;
    }
    if (lane == 0) {
      st.parent[r] = par;
      if (!frozen) st.run_score[r] = n_rs[k];
    }
  }
  if (frozen || !s_changed) return;
  for (int e = threadIdx.x; e < K * ML; e += blockDim.x) stage[e] = st.fin_ids[(size_t)row0 * ML + e];
  __syncthreads();
  for (int e = threadIdx.x; e < K * ML; e += blockDim.x) {
    const int k = e / ML, j = e % ML, src = f_src[k];
    int v;
    if (src < K) v = stage[src * ML + j];
    else {
      const int c = src - K;
      v = j < t ? st.ids_cur[(size_t)(row0 + s_beam[c]) * ML + j] : j == t ? s_tok[c] : st.pad_id;
    }
    st.fin_ids[(size_t)row0 * ML + e] = v;
  }
  // lengths before scores: the old values of moved slots are read here first
  __shared__ int o_len[8];
  if (threadIdx.x < K) o_len[threadIdx.x] = st.fin_len[row0 + threadIdx.x];
  __syncthreads();
  if (threadIdx.x < K) {
    const int k = threadIdx.x, src = f_src[k];
    st.fin_len[row0 + k] = src < K ? o_len[src] : t + 1;
    st.fin_score[row0 + k] = f_score[k];
    st.fin_flag[row0 + k] = f_flag[k];
  }
}

__global__ void beam_output_kernel(BeamState st, int nr, int32_t* __restrict__ out_ids, int32_t* __restrict__ out_len,
                                   float* __restrict__ out_score) {
  const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int ML = st.max_len;
  if (e >= (int64_t)st.n * nr * ML) return;
  const int j = (int)(e % ML);
  const int64_t h = e / ML;                          // sentence * nr + rank
  const int64_t r = h / nr * st.K + h % nr;          // finished slot row
  const int len = st.fin_len[r];
  out_ids[e] = j < len ? st.fin_ids[r * ML + j] : st.pad_id;
  if (j == 0) {
    out_len[h] = len;
    out_score[h] = st.fin_score[r];
  }
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
                            void* kv_cache, void* ctx, int rows, int H, int max_keys, bool fp16, cudaStream_t s,
                            const int32_t* slot) {
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
  if (slot && key_start) return fail(PLLB_ERR_INVALID, "decode_attention: a slot table needs the self form");
  if (slot) {
    if (fp16)
      decode_attention_kernel<true, true><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len, self_t,
                                                                  max_len, nk, new_kv_stride, kc, cc, rows, H, NH, max_keys,
                                                                  slot);
    else
      decode_attention_kernel<false, true><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len,
                                                                   self_t, max_len, nk, new_kv_stride, kc, cc, rows, H, NH,
                                                                   max_keys, slot);
  } else if (fp16)
    decode_attention_kernel<true, false><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len, self_t,
                                                                 max_len, nk, new_kv_stride, kc, cc, rows, H, NH, max_keys,
                                                                 nullptr);
  else
    decode_attention_kernel<false, false><<<grid, 128, smem, s>>>(qq, q_stride, kk, kv_stride, key_start, key_len, self_t,
                                                                  max_len, nk, new_kv_stride, kc, cc, rows, H, NH, max_keys,
                                                                  nullptr);
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

int launch_beam_init(BeamState st, cudaStream_t s) {
  const int rows = std::max(st.n * st.K, 1);
  beam_init_kernel<<<(unsigned)ceil_div(rows, 128), 128, 0, s>>>(st);
  PLLB_LAUNCH_CHECK("beam_init_kernel");
  return PLLB_OK;
}

int launch_beam_select(const float2* partials, int n_parts, int ksel, int vocab, BeamState st, int t, cudaStream_t s) {
  if (st.n <= 0) return PLLB_OK;
  if (st.K < 2 || 2 * st.K > ksel || st.K > 8) return fail(PLLB_ERR_INVALID, "beam_select: need 2 <= K <= 8, 2K <= ksel");
  const size_t smem = sizeof(int32_t) * (size_t)st.K * st.max_len;
  if (smem > 48 * 1024) return fail(PLLB_ERR_INVALID, "beam_select: num_beams * max_length > 12288");
  if (ksel == 8) beam_select_kernel<8><<<st.n, 256, smem, s>>>(partials, n_parts, vocab, st, t);
  else if (ksel == 16) beam_select_kernel<16><<<st.n, 256, smem, s>>>(partials, n_parts, vocab, st, t);
  else return fail(PLLB_ERR_INVALID, "beam_select: ksel must be 8 or 16");
  PLLB_LAUNCH_CHECK("beam_select_kernel");
  return PLLB_OK;
}

int launch_beam_output(BeamState st, int r, int32_t* out_ids, int32_t* out_len, float* out_score, cudaStream_t s) {
  const int64_t total = (int64_t)st.n * r * st.max_len;
  if (total <= 0) return PLLB_OK;
  beam_output_kernel<<<(unsigned)ceil_div(total, 256), 256, 0, s>>>(st, r, out_ids, out_len, out_score);
  PLLB_LAUNCH_CHECK("beam_output_kernel");
  return PLLB_OK;
}

}  // namespace pllb
