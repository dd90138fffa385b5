// rescore_kernels.cu — stage 4: the rescoring combiner and the Levenshtein CER kernel.
// Compiled with -fmad=false: the fp64 arithmetic must round exactly like numpy's
// elementwise ops in rescore.py:47-53 (no FMA contraction).
#include <algorithm>

#include "common.h"

namespace pllb {

namespace {

// (1-weight)*(am)/hyps_len + weight*(lm)/hyps_len evaluated as numpy does:
// (((1-w)*am)/len) + ((w*lm)/len), int64 len converted to float64 (rescore.py:51).
__device__ __forceinline__ double combine(double w, double am, double lm, double len, int variant) {
  const double one_minus_w = 1.0 - w;
  double a = one_minus_w * am;
  double l = w * lm;
  if (variant == 0) { a = a / len; l = l / len; }
  else if (variant == 2) { a = a / len; }
  return a + l;
}

// grid: (ceil(N/256), W).  One thread per (weight, utterance): scores of the n_best
// hypotheses, np.argmax semantics (first maximum, first NaN wins — rescore.py:56), then a
// block-level integer reduction of the chosen hypotheses' edit distances.
__global__ void rescore_sweep_kernel(const double* __restrict__ am, const double* __restrict__ lm,
                                     const int64_t* __restrict__ len, const int32_t* __restrict__ dist, int32_t N,
                                     int32_t n_best, const double* __restrict__ weights, int32_t variant,
                                     int32_t* __restrict__ out_argmax, unsigned long long* __restrict__ out_edit_sum) {
  const int wi = blockIdx.y;
  const int u = blockIdx.x * blockDim.x + threadIdx.x;
  const double w = weights[wi];
  long long my = 0;
  if (u < N) {
    const size_t base = (size_t)u * n_best;
    int best = 0;
    double bv = combine(w, am[base], lm[base], (double)len[base], variant);
    bool done = isnan(bv);
    for (int k = 1; k < n_best && !done; ++k) {
      const double v = combine(w, am[base + k], lm[base + k], (double)len[base + k], variant);
      if (isnan(v)) { best = k; done = true; }
      else if (v > bv) { bv = v; best = k; }
    }
    out_argmax[(size_t)wi * N + u] = best;
    my = dist ? dist[base + best] : 0;
  }
  // integer sums are associative: any reduction order gives the reference's count
  __shared__ long long red[8];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) my += __shfl_xor_sync(0xffffffffu, my, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = my;
  __syncthreads();
  if (threadIdx.x == 0 && out_edit_sum) {
    long long t = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    atomicAdd(out_edit_sum + wi, (unsigned long long)t);
  }
}

__global__ void rescore_scores_kernel(const double* __restrict__ am, const double* __restrict__ lm,
                                      const int64_t* __restrict__ len, int64_t n, double w, int32_t variant,
                                      double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = combine(w, am[i], lm[i], (double)len[i], variant);
}

// Warp-per-pair Levenshtein.  Lanes own columns (hypothesis characters, KB blocks of 32);
// rows (reference characters) are processed one at a time.  The in-row dependency
// D[i][j-1]+1 is resolved with a warp prefix-min:  D[i][j] = j + min_{k<=j}(t[k]-k) with
// t[k] = min(D[i-1][k-1]+cost, D[i-1][k]+1), t[0] = i.
template <int KB>
__global__ void levenshtein_kernel(const int32_t* __restrict__ ref_cp, const int64_t* __restrict__ ref_off,
                                   const int32_t* __restrict__ hyp_cp, const int64_t* __restrict__ hyp_off,
                                   const int32_t* __restrict__ pair_ref, int32_t n_pairs, int32_t* __restrict__ out) {
  const int pair = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (pair >= n_pairs) return;
  const int r = pair_ref[pair];
  const int32_t* a = ref_cp + ref_off[r];
  const int na = (int)(ref_off[r + 1] - ref_off[r]);
  const int32_t* b = hyp_cp + hyp_off[pair];
  const int nb = (int)(hyp_off[pair + 1] - hyp_off[pair]);
  int bc[KB], prev[KB];
#pragma unroll
  for (int k = 0; k < KB; ++k) {
    const int j = k * 32 + lane;
    bc[k] = (j < nb) ? b[j] : -1;
    prev[k] = j + 1;                       // D[0][j+1]
  }
  for (int i = 1; i <= na; ++i) {
    const int ai = a[i - 1];
    int carry_diag = i - 1;                // D[i-1][0]
    int carry_min = i;                     // D[i][0] - 0
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      if (k * 32 < nb) {
        const int j = k * 32 + lane + 1;
        const int up = prev[k];
        int diag = __shfl_up_sync(0xffffffffu, up, 1);
        if (lane == 0) diag = carry_diag;
        carry_diag = __shfl_sync(0xffffffffu, up, 31);
        const int t = min(diag + (ai != bc[k] ? 1 : 0), up + 1);
        int x = t - j;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int y = __shfl_up_sync(0xffffffffu, x, o);
          if (lane >= o) x = min(x, y);
        }
        x = min(x, carry_min);
        carry_min = __shfl_sync(0xffffffffu, x, 31);
        prev[k] = x + j;
      }
    }
  }
  int result = na;                          // nb == 0
#pragma unroll
  for (int k = 0; k < KB; ++k) {
    if (nb > 0 && (nb - 1) / 32 == k) result = __shfl_sync(0xffffffffu, prev[k], (nb - 1) & 31);
  }
  if (lane == 0) out[pair] = result;
}

// Edit-operation alignment (DESIGN.md §3.10).  The forward pass is levenshtein_kernel's row
// recurrence; at every cell it also decides the backtrace code with the priority
// diagonal (0 = U, 1 = S) > up (2 = I) > left (3 = D).  Diagonal and up are tested against the
// new value directly; when neither attains it, the left neighbour does.  The 2-bit codes of one
// (row, 32-column block) are two ballots, stored by lane 0 as one uint2: in shared memory when
// the pair fits 64 x 64 (1 KB per warp), otherwise in the warp's slot of a global scratch region.
// Lane 0 then walks the codes back from (na, nb), writing ops backwards to the end of the pair's
// slot; the warp moves them to the slot's start and zeroes the rest.  Warps loop over pairs,
// so the global slots bound the scratch whatever the pair count.
constexpr int kAlignWarps = 8;                 // warps per block
constexpr int kAlignSmemSide = 64;             // pairs with na, nb <= 64 keep their codes on chip
constexpr uint32_t kAlignLetters = 0x44495355u;  // 'U' 'S' 'I' 'D', code c in byte c

template <int KB>
__global__ void __launch_bounds__(kAlignWarps * 32)
align_kernel(const int32_t* __restrict__ ref_cp, const int64_t* __restrict__ ref_off,
             const int32_t* __restrict__ hyp_cp, const int64_t* __restrict__ hyp_off,
             const int32_t* __restrict__ pair_ref, int32_t n_pairs, int32_t max_ref, int32_t max_hyp,
             const int64_t* __restrict__ ops_off, uint8_t* __restrict__ out_ops, int32_t* __restrict__ out_n_ops,
             int32_t* __restrict__ out_counts, uint2* __restrict__ gcodes, int64_t slot_words) {
  __shared__ uint2 s_codes[kAlignWarps][kAlignSmemSide * (kAlignSmemSide / 32)];
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int gwarp = blockIdx.x * kAlignWarps + warp;
  for (int pair = gwarp; pair < n_pairs; pair += gridDim.x * kAlignWarps) {
    const int r = pair_ref[pair];
    const int32_t* a = ref_cp + ref_off[r];
    const int na = (int)(ref_off[r + 1] - ref_off[r]);
    const int32_t* b = hyp_cp + hyp_off[pair];
    const int nb = (int)(hyp_off[pair + 1] - hyp_off[pair]);
    const int64_t off = ops_off[pair];
    if (na > max_ref || nb > max_hyp) {       // longer than the launch was sized for
      if (lane == 0) {
        out_n_ops[pair] = -1;
        for (int c = 0; c < 4; ++c) out_counts[4 * (int64_t)pair + c] = 0;
      }
      continue;
    }
    const int nbk = (nb + 31) >> 5;
    uint2* codes = (na <= kAlignSmemSide && nb <= kAlignSmemSide) ? s_codes[warp] : gcodes + gwarp * slot_words;
    int bc[KB], prev[KB];
#pragma unroll
    for (int k = 0; k < KB; ++k) {
      const int j = k * 32 + lane;
      bc[k] = (j < nb) ? b[j] : -1;
      prev[k] = j + 1;                       // D[0][j+1]
    }
    for (int i = 1; i <= na; ++i) {
      const int ai = a[i - 1];
      uint2* row = codes + (i - 1) * nbk;
      int carry_diag = i - 1;                // D[i-1][0]
      int carry_min = i;                     // D[i][0] - 0
#pragma unroll
      for (int k = 0; k < KB; ++k) {
        if (k * 32 < nb) {
          const int j = k * 32 + lane + 1;
          const int up = prev[k];
          int diag = __shfl_up_sync(0xffffffffu, up, 1);
          if (lane == 0) diag = carry_diag;
          carry_diag = __shfl_sync(0xffffffffu, up, 31);
          const int sub = ai != bc[k] ? 1 : 0;
          const int dv = diag + sub;
          const int t = min(dv, up + 1);
          int x = t - j;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x = min(x, y);
          }
          x = min(x, carry_min);
          carry_min = __shfl_sync(0xffffffffu, x, 31);
          const int v = x + j;
          const int code = dv == v ? sub : (up + 1 == v ? 2 : 3);
          const uint32_t lo = __ballot_sync(0xffffffffu, code & 1);
          const uint32_t hi = __ballot_sync(0xffffffffu, code & 2);
          if (lane == 0) row[k] = make_uint2(lo, hi);
          prev[k] = v;
        }
      }
    }
    int n = 0;
    if (lane == 0) {                         // the walk reads only what this lane stored
      int i = na, j = nb;
      int64_t w = off + na + nb;
      uint64_t cnt = 0;                      // four 16-bit counters U, S, I, D
      while (i > 0 && j > 0) {
        const uint2 word = codes[(i - 1) * nbk + ((j - 1) >> 5)];
        const int sh = (j - 1) & 31;
        const int c = ((word.x >> sh) & 1) | (((word.y >> sh) & 1) << 1);
        out_ops[--w] = (uint8_t)(kAlignLetters >> (8 * c));
        cnt += 1ull << (16 * c);
        i -= c != 3;
        j -= c != 2;
      }
      for (; i > 0; --i) { out_ops[--w] = 'I'; cnt += 1ull << 32; }
      for (; j > 0; --j) { out_ops[--w] = 'D'; cnt += 1ull << 48; }
      n = (int)(off + na + nb - w);
      out_n_ops[pair] = n;
#pragma unroll
      for (int c = 0; c < 4; ++c) out_counts[4 * (int64_t)pair + c] = (int32_t)((cnt >> (16 * c)) & 0xffff);
    }
    n = __shfl_sync(0xffffffffu, n, 0);
    const int shift = na + nb - n;
    __syncwarp();
    // Move [off+shift, off+shift+n) to [off, off+n) in ascending 32-byte steps: a step's
    // stores end below the next step's loads because shift >= 0.
    for (int base = 0; base < n; base += 32) {
      const int p = base + lane;
      const uint8_t op = p < n ? out_ops[off + shift + p] : 0;
      __syncwarp();
      if (p < n) out_ops[off + p] = op;
      __syncwarp();
    }
    for (int p = n + lane; p < na + nb; p += 32) out_ops[off + p] = 0;
    __syncwarp();
  }
}

}  // namespace

// Warps of one align launch and the global code slot (uint2 words) of each; 0 words when every
// pair keeps its codes in shared memory.  The slots hold max_ref rows of ceil(max_hyp/32) words
// and, together, at most kAlignScratchBudget bytes (at least one block's worth).
constexpr int64_t kAlignScratchBudget = 256ll << 20;

void align_shape(int32_t n_pairs, int32_t max_ref, int32_t max_hyp, int32_t* warps, int64_t* slot_words) {
  const int64_t need = ceil_div((int64_t)n_pairs, kAlignWarps) * kAlignWarps;
  if (max_ref <= kAlignSmemSide && max_hyp <= kAlignSmemSide) {
    *warps = (int32_t)need;
    *slot_words = 0;
    return;
  }
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) {
    cudaGetLastError();
    sms = 148;
  }
  const int64_t words = (int64_t)std::max(max_ref, 1) * ceil_div((int64_t)std::max(max_hyp, 1), 32);
  int64_t w = std::min<int64_t>(need, (int64_t)sms * 2 * kAlignWarps);
  w = std::min<int64_t>(w, std::max<int64_t>(kAlignWarps, kAlignScratchBudget / (8 * words) / kAlignWarps * kAlignWarps));
  *warps = (int32_t)w;
  *slot_words = words;
}

int launch_align(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
                 const int32_t* pair_ref, int32_t n_pairs, int32_t max_ref, int32_t max_hyp, const int64_t* ops_off,
                 uint8_t* out_ops, int32_t* out_n_ops, int32_t* out_counts, uint2* gcodes, cudaStream_t s) {
  if (n_pairs <= 0) return PLLB_OK;
  if (max_ref < 0 || max_hyp < 0) return fail(PLLB_ERR_INVALID, "align: negative max length");
  if (max_ref > 1024 || max_hyp > 1024) return fail(PLLB_ERR_TOO_LONG, "align: a side longer than 1024 symbols");
  int32_t warps = 0;
  int64_t slot_words = 0;
  align_shape(n_pairs, max_ref, max_hyp, &warps, &slot_words);
  if (slot_words > 0 && !gcodes) return fail(PLLB_ERR_INVALID, "align: long pairs need a code scratch region");
  const unsigned grid = (unsigned)(warps / kAlignWarps);
#define ALIGN(KB)                                                                                             \
  align_kernel<KB><<<grid, kAlignWarps * 32, 0, s>>>(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref, n_pairs, max_ref, \
                                                     max_hyp, ops_off, out_ops, out_n_ops, out_counts, gcodes,  \
                                                     slot_words)
  if (max_hyp <= 32) ALIGN(1);
  else if (max_hyp <= 64) ALIGN(2);
  else if (max_hyp <= 128) ALIGN(4);
  else if (max_hyp <= 256) ALIGN(8);
  else if (max_hyp <= 512) ALIGN(16);
  else ALIGN(32);
#undef ALIGN
  PLLB_LAUNCH_CHECK("align_kernel");
  return PLLB_OK;
}

int launch_rescore_sweep(const double* am, const double* lm, const int64_t* len, const int32_t* dist, int32_t N,
                         int32_t n_best, const double* weights, int32_t W, int32_t variant, int32_t* out_argmax,
                         int64_t* out_edit_sum, cudaStream_t s) {
  if (N <= 0 || W <= 0) return PLLB_OK;
  if (n_best <= 0 || variant < 0 || variant > 2) return fail(PLLB_ERR_INVALID, "rescore_sweep: bad n_best/variant");
  if (out_edit_sum) PLLB_CUDA(cudaMemsetAsync(out_edit_sum, 0, sizeof(int64_t) * W, s));
  dim3 grid((unsigned)ceil_div(N, 256), (unsigned)W);
  rescore_sweep_kernel<<<grid, 256, 0, s>>>(am, lm, len, dist, N, n_best, weights, variant, out_argmax,
                                            reinterpret_cast<unsigned long long*>(out_edit_sum));
  PLLB_LAUNCH_CHECK("rescore_sweep_kernel");
  return PLLB_OK;
}

int launch_rescore_scores(const double* am, const double* lm, const int64_t* len, int32_t N, int32_t n_best,
                          double weight, int32_t variant, double* out, cudaStream_t s) {
  const int64_t n = (int64_t)N * n_best;
  if (n <= 0) return PLLB_OK;
  if (variant < 0 || variant > 2) return fail(PLLB_ERR_INVALID, "rescore_scores: bad variant");
  rescore_scores_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(am, lm, len, n, weight, variant, out);
  PLLB_LAUNCH_CHECK("rescore_scores_kernel");
  return PLLB_OK;
}

int launch_levenshtein(const int32_t* ref_cp, const int64_t* ref_off, const int32_t* hyp_cp, const int64_t* hyp_off,
                       const int32_t* pair_ref, int32_t n_pairs, int32_t max_len, int32_t* out, cudaStream_t s) {
  if (n_pairs <= 0) return PLLB_OK;
  const unsigned grid = (unsigned)ceil_div(n_pairs, 8);
#define LEV(KB) levenshtein_kernel<KB><<<grid, 256, 0, s>>>(ref_cp, ref_off, hyp_cp, hyp_off, pair_ref, n_pairs, out)
  if (max_len <= 32) LEV(1);
  else if (max_len <= 64) LEV(2);
  else if (max_len <= 128) LEV(4);
  else if (max_len <= 256) LEV(8);
  else if (max_len <= 512) LEV(16);
  else if (max_len <= 1024) LEV(32);
  else return fail(PLLB_ERR_TOO_LONG, "levenshtein: hypothesis longer than 1024 code points");
#undef LEV
  PLLB_LAUNCH_CHECK("levenshtein_kernel");
  return PLLB_OK;
}

}  // namespace pllb
