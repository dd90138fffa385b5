// encoder_kernels.cu — the HBM-bound pieces of the MLM-PLL path for sm_100a:
//   stage 1  masked-copy expansion with varlen packing (replaces MLM_PLL/preprocess.py:9-30
//            and the padded collate of MLM_PLL/main.py:28-54), fused with BertEmbeddings
//            (transformers modeling_bert.py:72-112);
//   the MLM head's LayerNorm (modeling_bert.py:481-487), per-sequence varlen
//            self-attention (:168-207), masked-row gather, logsumexp finish and the
//            per-hypothesis sum of MLM_PLL/main.py:101-107.
// All kernels are one-warp-per-row (or per sequence/head) with 128-bit accesses; rows of
// H fp32 are contiguous so every warp access is a fully coalesced 512-byte segment.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.h"
#include "ptx.cuh"

namespace pllb {

namespace {

constexpr int WARPS_PER_BLOCK = 8;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// two fp32 -> packed 16-bit pair in the operand dtype (bf16 or fp16); buffers are typed
// __nv_bfloat16 throughout and reinterpreted when the handle runs in fp16 mode.
template <bool FP16>
__device__ __forceinline__ uint32_t pack16(float lo, float hi) {
  return pack16x2_sat<FP16>(lo, hi);
}

// ---------------------------------------------------------------- plan
// One thread per hypothesis: writes the descriptors of its L masked copies.
__global__ void expand_plan_kernel(const int32_t* __restrict__ tokens, const int32_t* __restrict__ hyp_tok_off,
                                   const int32_t* __restrict__ hyp_copy_base, const int32_t* __restrict__ hyp_row_base,
                                   int32_t n_hyp, int32_t vocab, bool whole_sequence, CopyPlan plan) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= n_hyp) return;
  const int t0 = hyp_tok_off[h];
  const int L = hyp_tok_off[h + 1] - t0;
  const int T = L + 2;
  const int c0 = hyp_copy_base[h];
  const int r0 = hyp_row_base[h];
  if (whole_sequence) {
    // sequence-level scoring: ONE unmasked copy [CLS] t [SEP]; "mask_row" = the [CLS] row, so
    // copy_token_id never substitutes [MASK] (position 0 is [CLS]) and the last-layer pruning
    // gathers exactly the row the Linear(H,1) head reads (RescoreBert/model.py:19).
    plan.seq_start[c0] = r0;
    plan.seq_len[c0] = T;
    plan.mask_row[c0] = r0;
    plan.label[c0] = 0;
    plan.hyp[c0] = h;
    plan.uniq_base[c0] = 0;
    return;
  }
  for (int m = 0; m < L; ++m) {
    const int c = c0 + m;
    plan.seq_start[c] = r0 + m * T;
    plan.seq_len[c] = T;
    plan.mask_row[c] = r0 + m * T + m + 1;
    plan.label[c] = min(max(tokens[t0 + m], 0), vocab - 1);   // ids are validated on the host; clamp = memory safety
    plan.hyp[c] = h;
    plan.uniq_base[c] = 2 * t0 + 2 * h;                       // sum over earlier hypotheses of (T + L), see embed_unique_kernel
  }
}

__device__ __forceinline__ int copy_token_id(const int32_t* __restrict__ tokens, int t0, int T, int m, int p,
                                             int cls_id, int sep_id, int mask_id) {
  // [CLS] t[:m] [MASK] t[m+1:] [SEP] — MLM_PLL/preprocess.py:16-22
  if (p == 0) return cls_id;
  if (p == T - 1) return sep_id;
  if (p == m + 1) return mask_id;
  return tokens[t0 + p - 1];
}

// Materialises input_ids / mask_pos / labels (parity hook for stage 1; the scoring path
// never writes ids to HBM, see embed_ln_kernel).
__global__ void expand_ids_kernel(const int32_t* __restrict__ tokens, const int32_t* __restrict__ hyp_tok_off,
                                  CopyPlan plan, int32_t n_copies, int cls_id, int sep_id, int mask_id,
                                  int32_t* __restrict__ out_ids, int32_t* __restrict__ out_mask_pos,
                                  int32_t* __restrict__ out_labels) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n_copies) return;
  const int start = plan.seq_start[c], T = plan.seq_len[c];
  const int m = plan.mask_row[c] - start - 1;
  const int t0 = hyp_tok_off[plan.hyp[c]];
  for (int p = lane; p < T; p += 32) out_ids[start + p] = copy_token_id(tokens, t0, T, m, p, cls_id, sep_id, mask_id);
  if (lane == 0) {
    out_mask_pos[c] = m + 1;
    out_labels[c] = plan.label[c];
  }
}

// ---------------------------------------------------------------- LayerNorm helpers
// A warp owns one row of H = 128 * VEC floats; lane holds VEC float4 (columns 4*(lane+32*i)..).
template <int VEC>
__device__ __forceinline__ void ln_normalize(float4 (&x)[VEC], const float* __restrict__ g, const float* __restrict__ b,
                                             float eps, int lane) {
  constexpr float inv_h = 1.0f / (128.0f * VEC);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) s += (x[i].x + x[i].y) + (x[i].z + x[i].w);
  const float mean = warp_sum(s) * inv_h;
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float a = x[i].x - mean, bb = x[i].y - mean, c = x[i].z - mean, d = x[i].w - mean;
    v += (a * a + bb * bb) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(v) * inv_h + eps);
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + lane + 32 * i);
    const float4 be = __ldg(reinterpret_cast<const float4*>(b) + lane + 32 * i);
    x[i].x = (x[i].x - mean) * rstd * gg.x + be.x;
    x[i].y = (x[i].y - mean) * rstd * gg.y + be.y;
    x[i].z = (x[i].z - mean) * rstd * gg.z + be.z;
    x[i].w = (x[i].w - mean) * rstd * gg.w + be.w;
  }
}

// the row-major 16-bit copy of one row
template <int VEC, bool FP16>
__device__ __forceinline__ void store_row(const float4 (&x)[VEC], __nv_bfloat16* __restrict__ bf_row, int lane) {
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    if (bf_row) {
      uint2 u;
      u.x = pack16<FP16>(x[i].x, x[i].y);
      u.y = pack16<FP16>(x[i].z, x[i].w);
      reinterpret_cast<uint2*>(bf_row)[lane + 32 * i] = u;
    }
  }
}

// BertEmbeddings of one token (modeling_bert.py:72-112): (word + token_type(0)) + position -> LayerNorm.
template <int VEC>
__device__ __forceinline__ void embed_row(float4 (&x)[VEC], int id, int p, const float* __restrict__ word_emb,
                                          const float* __restrict__ pos_emb, const float* __restrict__ type_emb,
                                          const float* __restrict__ g, const float* __restrict__ b, float eps, int lane) {
  constexpr int H = 128 * VEC;
  const float4* w = reinterpret_cast<const float4*>(word_emb + (size_t)id * H);
  const float4* pe = reinterpret_cast<const float4*>(pos_emb + (size_t)p * H);
  const float4* te = reinterpret_cast<const float4*>(type_emb);
#pragma unroll
  for (int i = 0; i < VEC; ++i) {
    const float4 a = __ldg(w + lane + 32 * i), bb = __ldg(te + lane + 32 * i), cc = __ldg(pe + lane + 32 * i);
    // (word + token_type) + position — modeling_bert.py:104-108
    x[i].x = (a.x + bb.x) + cc.x; x[i].y = (a.y + bb.y) + cc.y;
    x[i].z = (a.z + bb.z) + cc.z; x[i].w = (a.w + bb.w) + cc.w;
  }
  ln_normalize<VEC>(x, g, b, eps, lane);
}

// ---------------------------------------------------------------- stage 1 + BertEmbeddings
// One warp per masked copy: derives every token id of the copy on the fly (ids never touch
// HBM), gathers word + position + token_type(0) rows, LayerNorm, writes the fp32 residual
// stream and the bf16 GEMM operand.
template <int VEC, bool FP16>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
embed_ln_kernel(const int32_t* __restrict__ tokens, const int32_t* __restrict__ hyp_tok_off, CopyPlan plan,
                int32_t n_copies, const float* __restrict__ word_emb, const float* __restrict__ pos_emb,
                const float* __restrict__ type_emb, const float* __restrict__ g, const float* __restrict__ b, float eps,
                int cls_id, int sep_id, int mask_id, int vocab, float* __restrict__ hidden_f32,
                __nv_bfloat16* __restrict__ hidden_bf16) {
  constexpr int H = 128 * VEC;
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n_copies) return;
  const int start = plan.seq_start[c], T = plan.seq_len[c];
  const int m = plan.mask_row[c] - start - 1;
  const int t0 = hyp_tok_off[plan.hyp[c]];
  for (int p = 0; p < T; ++p) {
    const int id = min(max(copy_token_id(tokens, t0, T, m, p, cls_id, sep_id, mask_id), 0), vocab - 1);
    float4 x[VEC];
    embed_row<VEC>(x, id, p, word_emb, pos_emb, type_emb, g, b, eps, lane);
    const size_t row = (size_t)(start + p);
    // fp32 goes out row-major here (one coalesced 3 KB row per warp); rowmajor_to_t32_kernel
    // re-tiles it into the T32 residual layout with fully coalesced accesses on both sides.
#pragma unroll
    for (int i = 0; i < VEC; ++i) reinterpret_cast<float4*>(hidden_f32 + row * H)[lane + 32 * i] = x[i];
    store_row<VEC, FP16>(x, hidden_bf16 + row * H, lane);
  }
}

// ---------------------------------------------------------------- layer-0 sharing
// The L masked copies of a hypothesis differ from the unmasked sequence [CLS] t [SEP] in ONE
// row each, and everything up to and including the layer-0 Q/K/V projection is row-wise.
// So embeddings and the layer-0 QKV GEMM run on the UNIQUE rows of a hypothesis only:
//   rows ub .. ub+T-1      the unmasked sequence, position p = row - ub
//   rows ub+T .. ub+T+L-1  [MASK] at position m+1, m = row - ub - T
// with ub = sum over earlier hypotheses of (T + L) = 2*tok_off + 2*h.  Row p of copy m maps to
// unique row (p == m+1 ? ub+T+m : ub+p).  Results are bit-identical to the per-copy path
// (same per-row arithmetic); 2L+2 rows instead of L(L+2).
constexpr int UNIQ_PARTS = 4;   // warps per hypothesis

template <int VEC, bool FP16>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
embed_unique_kernel(const int32_t* __restrict__ tokens, const int32_t* __restrict__ hyp_tok_off, int32_t n_hyp,
                    const float* __restrict__ word_emb, const float* __restrict__ pos_emb,
                    const float* __restrict__ type_emb, const float* __restrict__ g, const float* __restrict__ b,
                    float eps, int cls_id, int sep_id, int mask_id, int vocab, float* __restrict__ u_f32,
                    __nv_bfloat16* __restrict__ u_bf16) {
  constexpr int H = 128 * VEC;
  const int w = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const int h = w / UNIQ_PARTS, part = w % UNIQ_PARTS;
  if (h >= n_hyp) return;
  const int t0 = hyp_tok_off[h];
  const int L = hyp_tok_off[h + 1] - t0, T = L + 2;
  const size_t ub = (size_t)2 * t0 + 2 * h;
  for (int j = part; j < T + L; j += UNIQ_PARTS) {
    const int p = j < T ? j : j - T + 1;
    int id = j >= T ? mask_id : (p == 0 ? cls_id : (p == T - 1 ? sep_id : tokens[t0 + p - 1]));
    id = min(max(id, 0), vocab - 1);
    float4 x[VEC];
    embed_row<VEC>(x, id, p, word_emb, pos_emb, type_emb, g, b, eps, lane);
    const size_t row = ub + j;
#pragma unroll
    for (int i = 0; i < VEC; ++i) reinterpret_cast<float4*>(u_f32 + row * H)[lane + 32 * i] = x[i];
    store_row<VEC, FP16>(x, u_bf16 + row * H, lane);
  }
}

// row_src[packed row] = unique row it equals (one warp per copy)
__global__ void row_src_kernel(CopyPlan plan, int32_t n_copies) {
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n_copies) return;
  const int start = plan.seq_start[c], T = plan.seq_len[c], ub = plan.uniq_base[c];
  const int mpos = plan.mask_row[c] - start;
  for (int p = lane; p < T; p += 32) plan.row_src[start + p] = p == mpos ? ub + T + mpos - 1 : ub + p;
}

// out_bf16 = 16-bit(LayerNorm(y)), y row-major fp32.  One warp per row.
template <int VEC, bool FP16>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
ln_kernel(const float* __restrict__ y, __nv_bfloat16* __restrict__ out_bf16, const float* __restrict__ g,
          const float* __restrict__ b, float eps, int64_t rows) {
  constexpr int H = 128 * VEC;
  const int64_t row = (int64_t)blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* yr = reinterpret_cast<const float4*>(y + row * H);
  float4 x[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) x[i] = yr[lane + 32 * i];
  ln_normalize<VEC>(x, g, b, eps, lane);
  store_row<VEC, FP16>(x, out_bf16 + row * H, lane);
}

// ---------------------------------------------------------------- tensor-core varlen attention
// One warp per (masked copy, head), flash-style: 16-query tiles x 16-key blocks with an
// online softmax, S = Q K^T and O = P V on mma.sync.m16n8k16 (bf16 in, fp32 accumulate).
// Per-sequence tiles are 5..66 rows, far below the 128-row tcgen05 atom, and the two
// matmuls are 0.4 % of the path's FLOPs (SURVEY.md §8d): the warp-level MMA keeps every
// tile busy with no padding to 128 and leaves the kernel HBM-bound (6 KB per token).
// Q / K fragments are read straight from global memory (each element is used once per
// tile); V blocks are staged in shared memory and read with ldmatrix.trans.
constexpr int ATT_WARPS = 8;
constexpr int ATT_VROW = 72;   // bf16 elements per staged V row (144 B: conflict-free ldmatrix)

// 2^x on the SFU alone (MUFU.EX2; exp2f() wraps it in a range check and two scalings that the
// softmax does not need: its arguments are <= 0 and an underflow to 0 is the right answer).
__device__ __forceinline__ float fast_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

template <bool FP16>
__device__ __forceinline__ void mma_16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  if constexpr (FP16) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  } else {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
  }
}

// Packed row r of a sequence -> element offset of its [Q|K|V] row.  RowDirect: the copy's own rows;
// RowShared: the unique rows of its hypothesis (layer-0 sharing, see embed_unique_kernel).
struct RowDirect {
  size_t start_ld, ld;
  __device__ __forceinline__ size_t operator()(int r) const { return start_ld + (size_t)r * ld; }
};
struct RowShared {
  int ubase, umask, mpos;
  size_t ld;
  __device__ __forceinline__ size_t operator()(int r) const { return (size_t)(r == mpos ? umask : ubase + r) * ld; }
};

// Streaming form: any T; V blocks staged per 16-key block, Q/K fragments straight from global.
template <bool FP16, class RM>
__device__ __forceinline__ void attn_stream(const __nv_bfloat16* __restrict__ base /* qkv + head*64 */, const RM rm,
                                            __nv_bfloat16* __restrict__ ob, int T, int H, int lane, __nv_bfloat16* vs) {
  const __nv_bfloat16* kb = base + H;
  const __nv_bfloat16* vb = base + 2 * H;
  const int g = lane >> 2, cq = lane & 3;
  const uint32_t vs_addr = (uint32_t)__cvta_generic_to_shared(vs);
  constexpr float kScaleLog2 = 0.125f * 1.4426950408889634f;   // head_dim**-0.5 * log2(e)

  for (int m0 = 0; m0 < T; m0 += 16) {
    const size_t o0 = rm(min(m0 + g, T - 1)), o1 = rm(min(m0 + g + 8, T - 1));
    uint32_t qf[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      qf[ks][0] = *reinterpret_cast<const uint32_t*>(base + o0 + 16 * ks + 2 * cq);
      qf[ks][1] = *reinterpret_cast<const uint32_t*>(base + o1 + 16 * ks + 2 * cq);
      qf[ks][2] = *reinterpret_cast<const uint32_t*>(base + o0 + 16 * ks + 8 + 2 * cq);
      qf[ks][3] = *reinterpret_cast<const uint32_t*>(base + o1 + 16 * ks + 8 + 2 * cq);
    }
    float mx[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }

    for (int k0 = 0; k0 < T; k0 += 16) {
      // stage V[k0 .. k0+15][0..63] (rows clamped to T-1: masked keys get p = 0, values stay finite)
      __syncwarp();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = i * 4 + (lane >> 3), ch = lane & 7;
        const int key = min(k0 + row, T - 1);
        const uint4 v = *reinterpret_cast<const uint4*>(vb + rm(key) + ch * 8);
        *reinterpret_cast<uint4*>(vs + row * ATT_VROW + ch * 8) = v;
      }
      // S block = Q K^T for keys k0..k0+15 (two n-tiles of 8 keys)
      float s[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
        if (j == 1 && k0 + 8 >= T) break;               // second key tile fully masked (warp-uniform)
        const int key = min(k0 + 8 * j + g, T - 1);
        const __nv_bfloat16* kr = kb + rm(key) + 2 * cq;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint32_t b0 = *reinterpret_cast<const uint32_t*>(kr + 16 * ks);
          const uint32_t b1 = *reinterpret_cast<const uint32_t*>(kr + 16 * ks + 8);
          mma_16816<FP16>(s[j], qf[ks], b0, b1);
        }
      }
      // mask keys >= T, scale into the log2 domain, online softmax (rows g and g+8)
      float bm[2] = {-INFINITY, -INFINITY};
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = k0 + 8 * j + 2 * cq + (e & 1);
          s[j][e] = key < T ? s[j][e] * kScaleLog2 : -INFINITY;
          bm[e >> 1] = fmaxf(bm[e >> 1], s[j][e]);
        }
      }
      float corr[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        bm[r] = fmaxf(bm[r], __shfl_xor_sync(0xffffffffu, bm[r], 1));
        bm[r] = fmaxf(bm[r], __shfl_xor_sync(0xffffffffu, bm[r], 2));
        const float nm = fmaxf(mx[r], bm[r]);       // finite: every key block holds >= 1 valid key
        corr[r] = fast_ex2(mx[r] - nm);
        mx[r] = nm;
        l[r] *= corr[r];
      }
      uint32_t pf[4];
      {
        const float p00 = fast_ex2(s[0][0] - mx[0]), p01 = fast_ex2(s[0][1] - mx[0]);
        const float p02 = fast_ex2(s[0][2] - mx[1]), p03 = fast_ex2(s[0][3] - mx[1]);
        const float p10 = fast_ex2(s[1][0] - mx[0]), p11 = fast_ex2(s[1][1] - mx[0]);
        const float p12 = fast_ex2(s[1][2] - mx[1]), p13 = fast_ex2(s[1][3] - mx[1]);
        l[0] += (p00 + p01) + (p10 + p11);
        l[1] += (p02 + p03) + (p12 + p13);
        pf[0] = pack16<FP16>(p00, p01); pf[1] = pack16<FP16>(p02, p03);
        pf[2] = pack16<FP16>(p10, p11); pf[3] = pack16<FP16>(p12, p13);
      }
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        o[n][0] *= corr[0]; o[n][1] *= corr[0]; o[n][2] *= corr[1]; o[n][3] *= corr[1];
      }
      __syncwarp();   // V block visible to the whole warp
      // O += P V : 8 d-tiles of 8 columns, V^T fragments via ldmatrix.trans
#pragma unroll
      for (int n = 0; n < 8; n += 2) {
        const int mrow = (lane & 7) + ((lane >> 3) & 1) * 8;      // key row inside the block
        const int mcol = 8 * n + ((lane >> 4) & 1) * 8;           // d column of the 8x8 matrix
        const uint32_t addr = vs_addr + (uint32_t)(mrow * ATT_VROW + mcol) * 2;
        uint32_t b0, b1, b2, b3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
        mma_16816<FP16>(o[n], pf, b0, b1);
        mma_16816<FP16>(o[n + 1], pf, b2, b3);
      }
    }
    // finish: row sums across the quad, normalise, store bf16
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 1);
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 2);
    }
    const float inv0 = 1.0f / l[0], inv1 = 1.0f / l[1];
    const int q0 = m0 + g, q1 = m0 + g + 8;
#pragma unroll
    for (int n = 0; n < 8; ++n) {
      if (q0 < T)
        *reinterpret_cast<uint32_t*>(ob + (size_t)q0 * H + 8 * n + 2 * cq) = pack16<FP16>(o[n][0] * inv0, o[n][1] * inv0);
      if (q1 < T)
        *reinterpret_cast<uint32_t*>(ob + (size_t)q1 * H + 8 * n + 2 * cq) = pack16<FP16>(o[n][2] * inv1, o[n][3] * inv1);
    }
  }
}

// Staged form for T <= ATT_TS: the whole Q, K, V head slices of the sequence are brought
// into shared memory with one burst of cp.async (a single memory latency per sequence
// instead of one per 16x16 block), then every fragment comes from ldmatrix.
constexpr int ATT_TS = 32;
constexpr int ATT_STAGE_ELEMS = 3 * ATT_TS * ATT_VROW;   // bf16 elements per warp (13.5 KiB)

template <bool FP16, class RM>
__device__ __forceinline__ void attn_staged(const __nv_bfloat16* __restrict__ base /* qkv + head*64 */, const RM rm,
                                            __nv_bfloat16* __restrict__ ob, int T, int H, int lane, __nv_bfloat16* sm) {
  const int g = lane >> 2, cq = lane & 3;
  const uint32_t sm_addr = (uint32_t)__cvta_generic_to_shared(sm);
  constexpr float kScaleLog2 = 0.125f * 1.4426950408889634f;
  __syncwarp();                                           // previous sequence's fragments consumed
  {
    // 3 matrices x T rows x 8 chunks of 16 B; lane -> (row offset, chunk), no integer division
    const int r_off = lane >> 3, ch = lane & 7;
    for (int r = r_off; r < T; r += 4) {
      const __nv_bfloat16* src = base + rm(r) + ch * 8;
      const uint32_t dst = sm_addr + (uint32_t)(r * ATT_VROW + ch * 8) * 2;
#pragma unroll
      for (int mat = 0; mat < 3; ++mat)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)(mat * ATT_TS * ATT_VROW) * 2),
                     "l"(src + (size_t)mat * H) : "memory");
    }
    // V rows T .. ceil16(T)-1 are multiplied by p = 0: they must be finite (0 * NaN = NaN).  K / Q
    // padding rows only produce scores that are replaced by -inf / rows that are never stored.
    const int t16 = (T + 15) & ~15;
    for (int r = T + r_off; r < t16; r += 4)
      *reinterpret_cast<uint4*>(sm + (2 * ATT_TS + r) * ATT_VROW + ch * 8) = make_uint4(0, 0, 0, 0);
  }
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
  __syncwarp();
  const uint32_t q_addr = sm_addr, k_addr = sm_addr + ATT_TS * ATT_VROW * 2, v_addr = sm_addr + 2 * ATT_TS * ATT_VROW * 2;
  const int lrow = (lane & 7) + ((lane >> 3) & 1) * 8, lcol8 = ((lane >> 4) & 1) * 8;

  for (int m0 = 0; m0 < T; m0 += 16) {
    uint32_t qf[4][4];
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const uint32_t addr = q_addr + (uint32_t)((m0 + lrow) * ATT_VROW + 16 * ks + lcol8) * 2;
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                   : "=r"(qf[ks][0]), "=r"(qf[ks][1]), "=r"(qf[ks][2]), "=r"(qf[ks][3]) : "r"(addr));
    }
    float mx[2] = {-INFINITY, -INFINITY}, l[2] = {0.f, 0.f};
    float o[8][4];
#pragma unroll
    for (int n = 0; n < 8; ++n) { o[n][0] = o[n][1] = o[n][2] = o[n][3] = 0.f; }
    for (int k0 = 0; k0 < T; k0 += 16) {
      float s[2][4];
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
        if (j == 1 && k0 + 8 >= T) break;               // second key tile fully masked (warp-uniform)
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {                 // two k-steps per ldmatrix.x4
          const uint32_t addr = k_addr + (uint32_t)((k0 + 8 * j + (lane & 7)) * ATT_VROW + 32 * kp + (lane >> 3) * 8) * 2;
          uint32_t b0, b1, b2, b3;
          asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                       : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
          mma_16816<FP16>(s[j], qf[2 * kp], b0, b1);
          mma_16816<FP16>(s[j], qf[2 * kp + 1], b2, b3);
        }
      }
      float bm[2] = {-INFINITY, -INFINITY};
      const bool tail = k0 + 16 > T;                      // warp-uniform: only the last key block has padding keys
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int key = k0 + 8 * j + 2 * cq + (e & 1);
          s[j][e] = (!tail || key < T) ? s[j][e] * kScaleLog2 : -INFINITY;
          bm[e >> 1] = fmaxf(bm[e >> 1], s[j][e]);
        }
      }
      float corr[2];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        bm[r] = fmaxf(bm[r], __shfl_xor_sync(0xffffffffu, bm[r], 1));
        bm[r] = fmaxf(bm[r], __shfl_xor_sync(0xffffffffu, bm[r], 2));
        const float nm = fmaxf(mx[r], bm[r]);
        corr[r] = fast_ex2(mx[r] - nm);
        mx[r] = nm;
        l[r] *= corr[r];
      }
      uint32_t pf[4];
      {
        const float p00 = fast_ex2(s[0][0] - mx[0]), p01 = fast_ex2(s[0][1] - mx[0]);
        const float p02 = fast_ex2(s[0][2] - mx[1]), p03 = fast_ex2(s[0][3] - mx[1]);
        const float p10 = fast_ex2(s[1][0] - mx[0]), p11 = fast_ex2(s[1][1] - mx[0]);
        const float p12 = fast_ex2(s[1][2] - mx[1]), p13 = fast_ex2(s[1][3] - mx[1]);
        l[0] += (p00 + p01) + (p10 + p11);
        l[1] += (p02 + p03) + (p12 + p13);
        pf[0] = pack16<FP16>(p00, p01); pf[1] = pack16<FP16>(p02, p03);
        pf[2] = pack16<FP16>(p10, p11); pf[3] = pack16<FP16>(p12, p13);
      }
      if (k0 > 0) {
#pragma unroll
        for (int n = 0; n < 8; ++n) {
          o[n][0] *= corr[0]; o[n][1] *= corr[0]; o[n][2] *= corr[1]; o[n][3] *= corr[1];
        }
      }
#pragma unroll
      for (int n = 0; n < 8; n += 2) {
        const uint32_t addr = v_addr + (uint32_t)((k0 + lrow) * ATT_VROW + 8 * n + lcol8) * 2;
        uint32_t b0, b1, b2, b3;
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(b0), "=r"(b1), "=r"(b2), "=r"(b3) : "r"(addr));
        mma_16816<FP16>(o[n], pf, b0, b1);
        mma_16816<FP16>(o[n + 1], pf, b2, b3);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 1);
      l[r] += __shfl_xor_sync(0xffffffffu, l[r], 2);
    }
    const float inv0 = 1.0f / l[0], inv1 = 1.0f / l[1];
    // The Q rows of this block live in qf now: reuse them to transpose the context block so that
    // it leaves as 16-byte row-contiguous stores (4-byte fragment stores cost 8x the L1 wavefronts).
    __syncwarp();
    {
      const uint32_t st0 = q_addr + (uint32_t)((m0 + g) * ATT_VROW + 2 * cq) * 2, st1 = st0 + 8 * ATT_VROW * 2;
#pragma unroll
      for (int n = 0; n < 8; ++n) {
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(st0 + 16 * n), "r"(pack16<FP16>(o[n][0] * inv0, o[n][1] * inv0)) : "memory");
        asm volatile("st.shared.b32 [%0], %1;" ::"r"(st1 + 16 * n), "r"(pack16<FP16>(o[n][2] * inv1, o[n][3] * inv1)) : "memory");
      }
    }
    __syncwarp();
    {
      const int r_off = lane >> 3, ch = lane & 7;
#pragma unroll
      for (int rr = 0; rr < 16; rr += 4) {
        const int q = m0 + rr + r_off;
        if (q < T)
          *reinterpret_cast<uint4*>(ob + (size_t)q * H + ch * 8) =
              *reinterpret_cast<const uint4*>(sm + q * ATT_VROW + ch * 8);
      }
    }
  }
}

// SHARED: qkv holds the unique rows of every hypothesis (layer 0); otherwise one row per packed row.
template <bool FP16, bool SHARED>
__global__ void __launch_bounds__(ATT_WARPS * 32, 2)
attention_mma_kernel(const __nv_bfloat16* __restrict__ qkv, __nv_bfloat16* __restrict__ ctx, CopyPlan plan,
                     int32_t n_copies, int H, int NH) {
  extern __shared__ __align__(16) uint8_t att_dyn[];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __nv_bfloat16* sm = reinterpret_cast<__nv_bfloat16*>(att_dyn) + (size_t)wib * ATT_STAGE_ELEMS;
  const int64_t pair = (int64_t)blockIdx.x * ATT_WARPS + wib;
  if (pair >= (int64_t)n_copies * NH) return;
  const int c = (int)(pair / NH), head = (int)(pair % NH);
  const int start = plan.seq_start[c], T = plan.seq_len[c];
  const size_t ld = (size_t)3 * H;
  const __nv_bfloat16* base = qkv + head * 64;
  __nv_bfloat16* ob = ctx + (size_t)start * H + head * 64;
  if constexpr (SHARED) {
    const int ub = plan.uniq_base[c], mpos = plan.mask_row[c] - start;
    const RowShared rm{ub, ub + T + mpos - 1, mpos, ld};
    if (T <= ATT_TS) attn_staged<FP16>(base, rm, ob, T, H, lane, sm);
    else attn_stream<FP16>(base, rm, ob, T, H, lane, sm);
  } else {
    const RowDirect rm{(size_t)start * ld, ld};
    if (T <= ATT_TS) attn_staged<FP16>(base, rm, ob, T, H, lane, sm);
    else attn_stream<FP16>(base, rm, ob, T, H, lane, sm);
  }
}

// ---------------------------------------------------------------- last-layer attention
// Downstream of the last layer only ONE row per copy is consumed (the [MASK] row, or [CLS] for
// sequence scoring), so its attention has a single query row: q comes from the pruned Q
// projection [copies, H], K/V of the whole sequence from the K|V projection [rows, 2H].
// One warp per (copy, head): lane-per-key scores, fp32 softmax, lane-per-dimension-pair P·V.
constexpr int ATTR_MAXT = 512;

template <bool FP16>
__device__ __forceinline__ float2 unpack16(uint32_t u) {
  if constexpr (FP16) return __half22float2(*reinterpret_cast<const __half2*>(&u));
  else return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}

template <bool FP16>
__global__ void __launch_bounds__(WARPS_PER_BLOCK * 32)
attention_row_kernel(const __nv_bfloat16* __restrict__ q, const __nv_bfloat16* __restrict__ kv,
                     __nv_bfloat16* __restrict__ out, CopyPlan plan, int32_t n_copies, int H, int NH) {
  __shared__ float ps[WARPS_PER_BLOCK][ATTR_MAXT];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t pair = (int64_t)blockIdx.x * WARPS_PER_BLOCK + w;
  if (pair >= (int64_t)n_copies * NH) return;
  const int c = (int)(pair / NH), head = (int)(pair % NH);
  const int start = plan.seq_start[c], T = plan.seq_len[c];
  constexpr float kScaleLog2 = 0.125f * 1.4426950408889634f;   // head_dim**-0.5 * log2(e)
  // lane = (key slot r_off, 16-byte chunk ch): a warp access covers 4 rows x 128 contiguous bytes
  const int r_off = lane >> 3, ch = lane & 7;
  float qv[8];
  {
    const uint4 u = *reinterpret_cast<const uint4*>(q + (size_t)c * H + head * 64 + ch * 8);
    const float2 a = unpack16<FP16>(u.x), b = unpack16<FP16>(u.y), cc = unpack16<FP16>(u.z), d = unpack16<FP16>(u.w);
    qv[0] = a.x * kScaleLog2; qv[1] = a.y * kScaleLog2; qv[2] = b.x * kScaleLog2; qv[3] = b.y * kScaleLog2;
    qv[4] = cc.x * kScaleLog2; qv[5] = cc.y * kScaleLog2; qv[6] = d.x * kScaleLog2; qv[7] = d.y * kScaleLog2;
  }
  const size_t ld = (size_t)2 * H;
  const __nv_bfloat16* kb = kv + (size_t)start * ld + head * 64 + ch * 8;
  const __nv_bfloat16* vb = kb + H;
  float mx = -INFINITY;
  for (int j0 = 0; j0 < T; j0 += 4) {                       // warp-uniform trip count
    const int j = j0 + r_off;
    float sc = 0.f;
    if (j < T) {
      const uint4 u = *reinterpret_cast<const uint4*>(kb + (size_t)j * ld);
      const float2 a = unpack16<FP16>(u.x), b = unpack16<FP16>(u.y), cc = unpack16<FP16>(u.z), d = unpack16<FP16>(u.w);
      sc = (a.x * qv[0] + a.y * qv[1]) + (b.x * qv[2] + b.y * qv[3]) + (cc.x * qv[4] + cc.y * qv[5]) +
           (d.x * qv[6] + d.y * qv[7]);
    }
    sc += __shfl_xor_sync(0xffffffffu, sc, 1);
    sc += __shfl_xor_sync(0xffffffffu, sc, 2);
    sc += __shfl_xor_sync(0xffffffffu, sc, 4);
    if (j < T) {
      if (ch == 0) ps[w][j] = sc;
      mx = fmaxf(mx, sc);
    }
  }
  mx = warp_max(mx);
  __syncwarp();
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  float sum = 0.f;
  for (int j = r_off; j < T; j += 4) {
    const float pj = fast_ex2(ps[w][j] - mx);
    sum += pj;
    const uint4 u = *reinterpret_cast<const uint4*>(vb + (size_t)j * ld);
    const float2 a = unpack16<FP16>(u.x), b = unpack16<FP16>(u.y), cc = unpack16<FP16>(u.z), d = unpack16<FP16>(u.w);
    acc[0] += pj * a.x; acc[1] += pj * a.y; acc[2] += pj * b.x; acc[3] += pj * b.y;
    acc[4] += pj * cc.x; acc[5] += pj * cc.y; acc[6] += pj * d.x; acc[7] += pj * d.y;
  }
  // combine the four key slots (lanes with equal ch)
  sum += __shfl_xor_sync(0xffffffffu, sum, 8);
  sum += __shfl_xor_sync(0xffffffffu, sum, 16);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 8);
    acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 16);
  }
  if (r_off == 0) {
    const float inv = 1.0f / sum;
    uint4 o;
    o.x = pack16<FP16>(acc[0] * inv, acc[1] * inv);
    o.y = pack16<FP16>(acc[2] * inv, acc[3] * inv);
    o.z = pack16<FP16>(acc[4] * inv, acc[5] * inv);
    o.w = pack16<FP16>(acc[6] * inv, acc[7] * inv);
    *reinterpret_cast<uint4*>(out + (size_t)c * H + head * 64 + ch * 8) = o;
  }
}

// ---------------------------------------------------------------- head helpers
__global__ void gather_rows_bf16_kernel(const __nv_bfloat16* __restrict__ src, const int32_t* __restrict__ rows,
                                        int32_t n, int H, __nv_bfloat16* __restrict__ dst) {
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n) return;
  const uint4* s = reinterpret_cast<const uint4*>(src + (size_t)rows[c] * H);
  uint4* d = reinterpret_cast<uint4*>(dst + (size_t)c * H);
  for (int i = lane; i < H / 8; i += 32) d[i] = s[i];
}

__global__ void gather_rows_f32_kernel(const float* __restrict__ src, const int32_t* __restrict__ rows, int32_t n, int H,
                                       float* __restrict__ dst) {
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n) return;
  // both sides in the T32 blocked layout
  const int64_t sr = rows[c];
  const int G = H / 4;
  const float4* s = reinterpret_cast<const float4*>(src) + (size_t)(sr >> 5) * G * 32 + (sr & 31);
  float4* d = reinterpret_cast<float4*>(dst) + (size_t)(c >> 5) * G * 32 + (c & 31);
  for (int i = lane; i < G; i += 32) d[(size_t)i * 32] = s[(size_t)i * 32];
}

// row-major fp32 [rows, H] -> T32 blocked layout; one CTA per (32-row block, 128-column slab)
__global__ void __launch_bounds__(256)
rowmajor_to_t32_kernel(const float* __restrict__ src, const int32_t* __restrict__ row_src /* or null */,
                       float* __restrict__ dst, int64_t rows, int H) {
  __shared__ float tile[32][132];
  const int64_t r0 = (int64_t)blockIdx.x * 32;
  const int c0 = blockIdx.y * 128;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 4; ++k) {                               // warp w loads rows w, w+8, w+16, w+24 (512 B each)
    const int r = w + 8 * k;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (r0 + r < rows) {
      const int64_t sr = row_src ? (int64_t)row_src[r0 + r] : r0 + r;
      v = *reinterpret_cast<const float4*>(src + sr * H + c0 + 4 * lane);
    }
    *reinterpret_cast<float4*>(&tile[r][4 * lane]) = v;
  }
  __syncthreads();
  const int G = H / 4;
  float4* out = reinterpret_cast<float4*>(dst) + ((size_t)blockIdx.x * G + c0 / 4) * 32 + lane;
#pragma unroll
  for (int k = 0; k < 4; ++k) {                               // warp w writes column groups w, w+8, ... (512 B each)
    const int g = w + 8 * k;
    out[(size_t)g * 32] = *reinterpret_cast<const float4*>(&tile[lane][4 * g]);
  }
}

__global__ void t32_to_rowmajor_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t rows, int H) {
  const int64_t row = (int64_t)blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int G = H / 4;
  const float4* s = reinterpret_cast<const float4*>(src) + (size_t)(row >> 5) * G * 32 + (row & 31);
  float4* d = reinterpret_cast<float4*>(dst + row * H);
  for (int i = lane; i < G; i += 32) d[i] = s[(size_t)i * 32];
}

// out[c] = dot(hidden[c, :], w) + b on the T32-layout fp32 rows; one warp per row.
__global__ void cls_linear_kernel(const float* __restrict__ hid_t32, const float* __restrict__ w, float b, int32_t n, int H,
                                  float* __restrict__ out) {
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n) return;
  const int G = H / 4;
  const float4* row = reinterpret_cast<const float4*>(hid_t32) + (size_t)(c >> 5) * G * 32 + (c & 31);
  float acc = 0.f;
  for (int g = lane; g < G; g += 32) {
    const float4 x = row[(size_t)g * 32];
    const float4 ww = __ldg(reinterpret_cast<const float4*>(w) + g);
    acc += (x.x * ww.x + x.y * ww.y) + (x.z * ww.z + x.w * ww.w);
  }
  acc = warp_sum(acc);
  if (lane == 0) out[c] = acc + b;
}

// log_softmax(logits)[label] = label_logit - (max + log(sum exp)) — MLM_PLL/main.py:101-105
__global__ void lse_finish_kernel(const float2* __restrict__ partials, const float* __restrict__ label_logit,
                                  int32_t n_copies, int n_tiles, float* __restrict__ tok_logp) {
  const int c = blockIdx.x * WARPS_PER_BLOCK + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (c >= n_copies) return;
  const float2* pr = partials + (size_t)c * n_tiles;
  float m = -INFINITY;
  for (int t = lane; t < n_tiles; t += 32) m = fmaxf(m, pr[t].x);
  m = warp_max(m);
  float s = 0.f;
  for (int t = lane; t < n_tiles; t += 32) {
    const float2 v = pr[t];
    if (v.y > 0.f) s += v.y * expf(v.x - m);
  }
  s = warp_sum(s);
  if (lane == 0) tok_logp[c] = (label_logit[c] - m) - logf(s);
}

// output_score[u][h] += s over the L copies, in order, in double — MLM_PLL/main.py:106-107
__global__ void hyp_sum_kernel(const float* __restrict__ tok_logp, const int32_t* __restrict__ hyp_copy_base,
                               int32_t n_hyp, double* __restrict__ out_pll, float* __restrict__ out_tok_logp) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= n_hyp) return;
  const int c0 = hyp_copy_base[h], c1 = hyp_copy_base[h + 1];
  double acc = 0.0;
  for (int c = c0; c < c1; ++c) {
    const float v = tok_logp[c];
    acc += (double)v;
    if (out_tok_logp) out_tok_logp[c] = v;
  }
  out_pll[h] = acc;
}

template <bool FP16>
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(src + i);
    uint2 u;
    u.x = pack16<FP16>(v.x, v.y);
    u.y = pack16<FP16>(v.z, v.w);
    *reinterpret_cast<uint2*>(dst + i) = u;
  } else {
    for (int64_t j = i; j < n; ++j) {
      reinterpret_cast<uint16_t*>(dst)[j] = (uint16_t)(pack16<FP16>(src[j], 0.f) & 0xffffu);
    }
  }
}

}  // namespace

// ------------------------------------------------------------------ launchers
int launch_expand_plan(const int32_t* tokens, const int32_t* hyp_tok_off, const int32_t* hyp_copy_base,
                       const int32_t* hyp_row_base, int32_t n_hyp, int32_t vocab, bool whole_sequence, CopyPlan plan,
                       cudaStream_t s) {
  if (n_hyp <= 0) return PLLB_OK;
  expand_plan_kernel<<<(unsigned)ceil_div(n_hyp, 128), 128, 0, s>>>(tokens, hyp_tok_off, hyp_copy_base, hyp_row_base,
                                                                   n_hyp, vocab, whole_sequence, plan);
  PLLB_LAUNCH_CHECK("expand_plan_kernel");
  return PLLB_OK;
}

int launch_expand_ids(const int32_t* tokens, const int32_t* hyp_tok_off, CopyPlan plan, int32_t n_copies,
                      int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t* out_ids, int32_t* out_mask_pos,
                      int32_t* out_labels, cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  expand_ids_kernel<<<(unsigned)ceil_div(n_copies, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(
      tokens, hyp_tok_off, plan, n_copies, cls_id, sep_id, mask_id, out_ids, out_mask_pos, out_labels);
  PLLB_LAUNCH_CHECK("expand_ids_kernel");
  return PLLB_OK;
}

#define PLLB_DISPATCH_VEC(H, CALL)                                                   \
  switch ((H) / 128) {                                                               \
    case 2: { constexpr int VEC = 2; CALL; } break;                                  \
    case 4: { constexpr int VEC = 4; CALL; } break;                                  \
    case 6: { constexpr int VEC = 6; CALL; } break;                                  \
    case 8: { constexpr int VEC = 8; CALL; } break;                                  \
    default: return fail(PLLB_ERR_INVALID, "hidden size must be 256, 512, 768 or 1024"); \
  }

int launch_embed_ln(const int32_t* tokens, const int32_t* hyp_tok_off, CopyPlan plan, int32_t n_copies,
                    const float* word_emb, const float* pos_emb, const float* type_emb, const float* g, const float* b,
                    float eps, int H, int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t vocab, float* hidden_f32,
                    void* hidden_bf16, bool fp16, cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  const unsigned grid = (unsigned)ceil_div(n_copies, WARPS_PER_BLOCK);
#define EMB(F) embed_ln_kernel<VEC, F><<<grid, WARPS_PER_BLOCK * 32, 0, s>>>(                                         \
      tokens, hyp_tok_off, plan, n_copies, word_emb, pos_emb, type_emb, g, b, eps, cls_id, sep_id, mask_id, vocab,       \
      hidden_f32,                                                                                                      \
      reinterpret_cast<__nv_bfloat16*>(hidden_bf16))
  PLLB_DISPATCH_VEC(H, (fp16 ? EMB(true) : EMB(false)));
#undef EMB
  PLLB_LAUNCH_CHECK("embed_ln_kernel");
  return PLLB_OK;
}

int launch_embed_unique(const int32_t* tokens, const int32_t* hyp_tok_off, int32_t n_hyp, const float* word_emb,
                        const float* pos_emb, const float* type_emb, const float* g, const float* b, float eps, int H,
                        int32_t cls_id, int32_t sep_id, int32_t mask_id, int32_t vocab, float* u_f32, void* u_bf16,
                        bool fp16, cudaStream_t s) {
  if (n_hyp <= 0) return PLLB_OK;
  const unsigned grid = (unsigned)ceil_div((int64_t)n_hyp * UNIQ_PARTS, WARPS_PER_BLOCK);
#define EMU(F) embed_unique_kernel<VEC, F><<<grid, WARPS_PER_BLOCK * 32, 0, s>>>(                                      \
      tokens, hyp_tok_off, n_hyp, word_emb, pos_emb, type_emb, g, b, eps, cls_id, sep_id, mask_id, vocab, u_f32,         \
      reinterpret_cast<__nv_bfloat16*>(u_bf16))
  PLLB_DISPATCH_VEC(H, (fp16 ? EMU(true) : EMU(false)));
#undef EMU
  PLLB_LAUNCH_CHECK("embed_unique_kernel");
  return PLLB_OK;
}

int launch_row_src(CopyPlan plan, int32_t n_copies, cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  row_src_kernel<<<(unsigned)ceil_div(n_copies, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(plan, n_copies);
  PLLB_LAUNCH_CHECK("row_src_kernel");
  return PLLB_OK;
}

int launch_plain_ln_bf16(const float* x, void* out_bf16, const float* g, const float* b, float eps, int64_t rows, int H,
                         bool fp16, cudaStream_t s) {
  if (rows <= 0) return PLLB_OK;
  const unsigned grid = (unsigned)ceil_div(rows, WARPS_PER_BLOCK);
#define LNP(F) ln_kernel<VEC, F><<<grid, WARPS_PER_BLOCK * 32, 0, s>>>(                                        \
      x, reinterpret_cast<__nv_bfloat16*>(out_bf16), g, b, eps, rows)
  PLLB_DISPATCH_VEC(H, (fp16 ? LNP(true) : LNP(false)));
#undef LNP
  PLLB_LAUNCH_CHECK("ln_kernel<plain>");
  return PLLB_OK;
}

int launch_attention(const void* qkv_bf16, void* ctx_bf16, CopyPlan plan, int32_t n_copies, int H, int NH, bool fp16,
                     bool shared_rows, cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  if (H != NH * 64) return fail(PLLB_ERR_INVALID, "attention: head dim must be 64");
  const int64_t pairs = (int64_t)n_copies * NH;
  const int smem = ATT_WARPS * ATT_STAGE_ELEMS * 2;
  const unsigned grid = (unsigned)ceil_div(pairs, ATT_WARPS);
#define ATT(F, S)                                                                                                  \
  do {                                                                                                             \
    PLLB_CUDA(opt_in_smem(attention_mma_kernel<F, S>, smem));                                                      \
    attention_mma_kernel<F, S><<<grid, ATT_WARPS * 32, smem, s>>>(reinterpret_cast<const __nv_bfloat16*>(qkv_bf16), \
                                                                  reinterpret_cast<__nv_bfloat16*>(ctx_bf16), plan, \
                                                                  n_copies, H, NH);                                \
  } while (0)
  if (fp16) { if (shared_rows) ATT(true, true); else ATT(true, false); }
  else { if (shared_rows) ATT(false, true); else ATT(false, false); }
#undef ATT
  PLLB_LAUNCH_CHECK("attention_mma_kernel");
  return PLLB_OK;
}

int launch_attention_row(const void* q_bf16, const void* kv_bf16, void* out_bf16, CopyPlan plan, int32_t n_copies, int H,
                         int NH, int max_T, bool fp16, cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  if (H != NH * 64) return fail(PLLB_ERR_INVALID, "attention: head dim must be 64");
  if (max_T > ATTR_MAXT) return fail(PLLB_ERR_TOO_LONG, "attention_row: sequence longer than 512 rows");
  const unsigned grid = (unsigned)ceil_div((int64_t)n_copies * NH, WARPS_PER_BLOCK);
  if (fp16)
    attention_row_kernel<true><<<grid, WARPS_PER_BLOCK * 32, 0, s>>>(
        reinterpret_cast<const __nv_bfloat16*>(q_bf16), reinterpret_cast<const __nv_bfloat16*>(kv_bf16),
        reinterpret_cast<__nv_bfloat16*>(out_bf16), plan, n_copies, H, NH);
  else
    attention_row_kernel<false><<<grid, WARPS_PER_BLOCK * 32, 0, s>>>(
        reinterpret_cast<const __nv_bfloat16*>(q_bf16), reinterpret_cast<const __nv_bfloat16*>(kv_bf16),
        reinterpret_cast<__nv_bfloat16*>(out_bf16), plan, n_copies, H, NH);
  PLLB_LAUNCH_CHECK("attention_row_kernel");
  return PLLB_OK;
}

int launch_gather_rows_bf16(const void* hidden_bf16, const int32_t* rows, int32_t n, int H, void* out, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  gather_rows_bf16_kernel<<<(unsigned)ceil_div(n, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(
      reinterpret_cast<const __nv_bfloat16*>(hidden_bf16), rows, n, H, reinterpret_cast<__nv_bfloat16*>(out));
  PLLB_LAUNCH_CHECK("gather_rows_bf16_kernel");
  return PLLB_OK;
}

int launch_gather_rows_f32(const float* src, const int32_t* rows, int32_t n, int H, float* out, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  gather_rows_f32_kernel<<<(unsigned)ceil_div(n, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(src, rows, n, H, out);
  PLLB_LAUNCH_CHECK("gather_rows_f32_kernel");
  return PLLB_OK;
}

int launch_cls_linear(const float* hid_t32, const float* w, float b, int32_t n, int H, float* out, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  cls_linear_kernel<<<(unsigned)ceil_div(n, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(hid_t32, w, b, n, H, out);
  PLLB_LAUNCH_CHECK("cls_linear_kernel");
  return PLLB_OK;
}

int launch_lse_finish(const float2* partials, const float* label_logit, int32_t n_copies, int n_tiles, float* tok_logp,
                      cudaStream_t s) {
  if (n_copies <= 0) return PLLB_OK;
  lse_finish_kernel<<<(unsigned)ceil_div(n_copies, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(
      partials, label_logit, n_copies, n_tiles, tok_logp);
  PLLB_LAUNCH_CHECK("lse_finish_kernel");
  return PLLB_OK;
}

int launch_hyp_sum(const float* tok_logp, const int32_t* hyp_copy_base, int32_t n_hyp, double* out_pll,
                   float* out_tok_logp, cudaStream_t s) {
  if (n_hyp <= 0) return PLLB_OK;
  hyp_sum_kernel<<<(unsigned)ceil_div(n_hyp, 128), 128, 0, s>>>(tok_logp, hyp_copy_base, n_hyp, out_pll, out_tok_logp);
  PLLB_LAUNCH_CHECK("hyp_sum_kernel");
  return PLLB_OK;
}

int launch_rowmajor_to_t32(const float* src, const int32_t* row_src, float* dst, int64_t rows, int H, cudaStream_t s) {
  if (rows <= 0) return PLLB_OK;
  if (H % 128 != 0) return fail(PLLB_ERR_INVALID, "rowmajor_to_t32: H % 128 != 0");
  dim3 grid((unsigned)ceil_div(rows, 32), (unsigned)(H / 128));
  rowmajor_to_t32_kernel<<<grid, 256, 0, s>>>(src, row_src, dst, rows, H);
  PLLB_LAUNCH_CHECK("rowmajor_to_t32_kernel");
  return PLLB_OK;
}

int launch_t32_to_rowmajor(const float* src, float* dst, int64_t rows, int H, cudaStream_t s) {
  if (rows <= 0) return PLLB_OK;
  t32_to_rowmajor_kernel<<<(unsigned)ceil_div(rows, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(src, dst, rows, H);
  PLLB_LAUNCH_CHECK("t32_to_rowmajor_kernel");
  return PLLB_OK;
}

int launch_f32_to_bf16(const float* src, void* dst, int64_t n, bool fp16, cudaStream_t s) {
  if (n <= 0) return PLLB_OK;
  const unsigned grid = (unsigned)ceil_div(ceil_div(n, 4), 256);
  if (fp16) f32_to_bf16_kernel<true><<<grid, 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  else f32_to_bf16_kernel<false><<<grid, 256, 0, s>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), n);
  PLLB_LAUNCH_CHECK("f32_to_bf16_kernel");
  return PLLB_OK;
}

// ---------------------------------------------------------------------------------------------
// Text front end (SURVEY.md §8f rank 1): code points -> wordpiece ids for hypotheses made of
// CJK ideographs, punctuation and whitespace — BertTokenizer.tokenize + convert_tokens_to_ids at
// MLM_PLL/preprocess.py:10,16-27 (BasicTokenizer makes every such character its own token, so
// the mapping is a table lookup).  table[cp] >= 0: id; -1 whitespace (dropped); -2 removed
// (control, U+0000, U+FFFD); -3 part of a word run -> the whole hypothesis is flagged for the
// host wordpiece tokenizer and gets 0 tokens here.  One warp per hypothesis.
__device__ __forceinline__ int tok_lookup(const int32_t* __restrict__ table, int table_size, int32_t c) {
  return (c >= 0 && c < table_size) ? __ldg(table + c) : -3;
}

__global__ void tokenize_count_kernel(const int32_t* __restrict__ table, int table_size, const int32_t* __restrict__ cp,
                                      const int64_t* __restrict__ cp_off, int32_t n_hyp, int32_t* __restrict__ counts,
                                      uint8_t* __restrict__ needs_host) {
  const int h = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (h >= n_hyp) return;
  const int64_t b = cp_off[h], e = cp_off[h + 1];
  int n = 0, word = 0;
  for (int64_t i = b + lane; i < e; i += 32) {
    const int t = tok_lookup(table, table_size, cp[i]);
    n += t >= 0;
    word |= t == -3;
  }
  n = __reduce_add_sync(0xffffffffu, n);
  word = __any_sync(0xffffffffu, word);
  if (lane == 0) {
    counts[h] = word ? 0 : n;
    needs_host[h] = (uint8_t)word;
  }
}

__global__ void tokenize_write_kernel(const int32_t* __restrict__ table, int table_size, const int32_t* __restrict__ cp,
                                      const int64_t* __restrict__ cp_off, int32_t n_hyp,
                                      const uint8_t* __restrict__ needs_host, const int64_t* __restrict__ out_off,
                                      int32_t* __restrict__ out_ids) {
  const int h = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (h >= n_hyp || needs_host[h]) return;
  const int64_t b = cp_off[h], e = cp_off[h + 1];
  int64_t o = out_off[h];
  for (int64_t i0 = b; i0 < e; i0 += 32) {                    // warp-uniform trip count
    const int64_t i = i0 + lane;
    const int t = i < e ? tok_lookup(table, table_size, cp[i]) : -1;
    const unsigned keep = __ballot_sync(0xffffffffu, t >= 0);
    if (t >= 0) out_ids[o + __popc(keep & ((1u << lane) - 1u))] = t;
    o += __popc(keep);
  }
}

int launch_tokenize_count(const int32_t* table, int table_size, const int32_t* cp, const int64_t* cp_off, int32_t n_hyp,
                          int32_t* counts, uint8_t* needs_host, cudaStream_t s) {
  if (n_hyp <= 0) return PLLB_OK;
  tokenize_count_kernel<<<(unsigned)ceil_div((int64_t)n_hyp, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(
      table, table_size, cp, cp_off, n_hyp, counts, needs_host);
  PLLB_LAUNCH_CHECK("tokenize_count_kernel");
  return PLLB_OK;
}

int launch_tokenize_write(const int32_t* table, int table_size, const int32_t* cp, const int64_t* cp_off, int32_t n_hyp,
                          const uint8_t* needs_host, const int64_t* out_off, int32_t* out_ids, cudaStream_t s) {
  if (n_hyp <= 0) return PLLB_OK;
  tokenize_write_kernel<<<(unsigned)ceil_div((int64_t)n_hyp, WARPS_PER_BLOCK), WARPS_PER_BLOCK * 32, 0, s>>>(
      table, table_size, cp, cp_off, n_hyp, needs_host, out_off, out_ids);
  PLLB_LAUNCH_CHECK("tokenize_write_kernel");
  return PLLB_OK;
}

}  // namespace pllb
