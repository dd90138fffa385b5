// bertscore_kernels.cu — BERTScore recall of candidate/reference sentence pairs (RMBR's utility,
// include/pllb.h pllb_bertscore, DESIGN.md §3.9).
//
//   R(c, r) = mean over interior rows x of r (1 .. T_r-2) of max over ALL rows y of c of cos(E_r[x], E_c[y])
//   R = 0 when either sentence is empty (T == 2).
//
// One cooperative launch:
//   phase 1  every row's inverse L2 norm, once (warp per row, fixed-order lane sums + butterfly);
//   grid sync;
//   phase 2  one CTA per candidate group (a run of consecutive pairs with the same candidate, which is
//            how mbr_decode emits its pairs).  The candidate's rows (up to BS_CT at a time) sit in
//            shared memory while the CTA walks the interior rows of all the group's references in
//            tiles of BS_MT rows, streamed in K-slabs of BS_KS columns.  Each thread owns 2 reference
//            rows x up to 4 candidate rows; candidate values are warp-uniform (shared-memory
//            broadcast).  Every dot product is a sequential fp32 FMA chain over k, every max and sum
//            runs in a fixed order and nothing is atomic, so results are bit-deterministic.
#include <cooperative_groups.h>

#include <cfloat>

#include "common.h"

namespace cg = cooperative_groups;

namespace pllb {
namespace {

constexpr int BS_THREADS = 256;
constexpr int BS_WARPS = BS_THREADS / 32;
constexpr int BS_MT = 64;                 // reference rows per tile (2 per lane)
constexpr int BS_CQ = 4;                  // candidate rows per warp per chunk
constexpr int BS_CT = BS_WARPS * BS_CQ;   // candidate rows resident in shared memory (32)
constexpr int BS_KS = 32;                 // K-slab of the reference tile (floats)
constexpr int BS_RPAD = BS_KS + 4;        // row stride of the reference slab: conflict-free LDS.128

struct BsArgs {
  const float* emb;         // [rows, H] fp32 row-major
  const int32_t* row_off;   // [n_seq + 1] first row of each sequence
  const int32_t* pair_ref;  // [n_pairs] reference sequence of each pair
  const int32_t* item_off;  // [n_pairs + 1] prefix of the interior reference rows of the pairs
  const int32_t* grp_pair;  // [n_groups + 1] first pair of each candidate group
  const int32_t* grp_cand;  // [n_groups] candidate sequence of each group
  float* inv_norm;          // [rows - row_off[0]] scratch
  float* out;               // [n_pairs]
  int32_t n_groups, H;
  int32_t row_begin, row_end;
};

__device__ __forceinline__ void fma4(float& acc, const float4& a, const float4& b) {
  acc = fmaf(a.x, b.x, acc);
  acc = fmaf(a.y, b.y, acc);
  acc = fmaf(a.z, b.z, acc);
  acc = fmaf(a.w, b.w, acc);
}

__global__ void __launch_bounds__(BS_THREADS) bertscore_recall_kernel(BsArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int H = a.H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* cand_s = smem;                                   // [BS_CT][H]
  float* ref_s = cand_s + (size_t)BS_CT * H;              // [BS_MT][BS_RPAD]
  float* red_s = ref_s + BS_MT * BS_RPAD;                 // [BS_WARPS][BS_MT]
  float* best_s = red_s + BS_WARPS * BS_MT;               // [BS_MT] running max over candidate chunks
  float* cinv_s = best_s + BS_MT;                         // [BS_CT]
  int* item_row = reinterpret_cast<int*>(cinv_s + BS_CT); // [BS_MT] absolute row of each tile row
  int* item_pair = item_row + BS_MT;                      // [BS_MT] pair of each tile row

  // ---- phase 1: inverse norms, one warp per row
  {
    const int gw = (blockIdx.x * BS_THREADS + threadIdx.x) >> 5;
    const int nw = (gridDim.x * BS_THREADS) >> 5;
    for (int r = a.row_begin + gw; r < a.row_end; r += nw) {
      const float4* x = reinterpret_cast<const float4*>(a.emb + (size_t)r * H);
      float ss = 0.f;
      for (int k = lane; k < H / 4; k += 32) fma4(ss, x[k], x[k]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
      if (lane == 0) a.inv_norm[r - a.row_begin] = 1.0f / sqrtf(ss);
    }
  }
  cg::this_grid().sync();

  // ---- phase 2: one candidate group per CTA iteration
  for (int g = blockIdx.x; g < a.n_groups; g += gridDim.x) {
    const int p0 = a.grp_pair[g], p1 = a.grp_pair[g + 1];
    const int c = a.grp_cand[g];
    const int c_row = a.row_off[c], Tc = a.row_off[c + 1] - c_row;
    const int i_begin = a.item_off[p0], i_end = a.item_off[p1];
    // pairs without interior reference rows, or with an empty candidate, are 0 by definition
    for (int p = p0 + threadIdx.x; p < p1; p += BS_THREADS)
      if (Tc <= 2 || a.item_off[p + 1] == a.item_off[p]) a.out[p] = 0.f;
    if (Tc <= 2 || i_end == i_begin) continue;
    const int n_chunks = (Tc + BS_CT - 1) / BS_CT;
    float run_sum = 0.f;          // thread 0: sum of the current pair's row maxima, in row order
    for (int t0 = i_begin; t0 < i_end; t0 += BS_MT) {
      const int nt = min(BS_MT, i_end - t0);
      __syncthreads();            // previous tile's item_row / best_s readers are done
      if (threadIdx.x < BS_MT) {
        const int it = t0 + threadIdx.x;
        int row = -1, pp = -1;
        if (threadIdx.x < nt) {
          int lo = p0, hi = p1 - 1;   // last pair with item_off[p] <= it
          while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (a.item_off[mid] <= it) lo = mid; else hi = mid - 1;
          }
          pp = lo;
          row = a.row_off[a.pair_ref[lo]] + 1 + (it - a.item_off[lo]);
        }
        item_row[threadIdx.x] = row;
        item_pair[threadIdx.x] = pp;
        best_s[threadIdx.x] = -FLT_MAX;
      }
      for (int ch = 0; ch < n_chunks; ++ch) {
        const int cr0 = ch * BS_CT, ct = min(BS_CT, Tc - cr0);
        if (n_chunks > 1 || t0 == i_begin) {      // a single chunk stays resident for the whole group
          __syncthreads();
          const float4* src = reinterpret_cast<const float4*>(a.emb + (size_t)(c_row + cr0) * H);
          float4* dst = reinterpret_cast<float4*>(cand_s);
          for (int i = threadIdx.x; i < ct * (H / 4); i += BS_THREADS) dst[i] = src[i];
          if (threadIdx.x < ct) cinv_s[threadIdx.x] = a.inv_norm[c_row + cr0 + threadIdx.x - a.row_begin];
        }
        float acc[2][BS_CQ];
#pragma unroll
        for (int m = 0; m < 2; ++m)
#pragma unroll
          for (int q = 0; q < BS_CQ; ++q) acc[m][q] = 0.f;
        for (int k0 = 0; k0 < H; k0 += BS_KS) {
          __syncthreads();
          // reference slab [BS_MT][BS_KS]: 8 float4 per row, 512 float4 per slab, 2 per thread
#pragma unroll
          for (int rep = 0; rep < (BS_MT * BS_KS / 4) / BS_THREADS; ++rep) {
            const int idx = threadIdx.x + rep * BS_THREADS;
            const int m = idx / (BS_KS / 4), kq = idx % (BS_KS / 4);
            const int row = item_row[m];
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row >= 0) v = *reinterpret_cast<const float4*>(a.emb + (size_t)row * H + k0 + 4 * kq);
            *reinterpret_cast<float4*>(ref_s + m * BS_RPAD + 4 * kq) = v;
          }
          __syncthreads();
#pragma unroll
          for (int kk = 0; kk < BS_KS; kk += 4) {
            const float4 r0 = *reinterpret_cast<const float4*>(ref_s + lane * BS_RPAD + kk);
            const float4 r1 = *reinterpret_cast<const float4*>(ref_s + (lane + 32) * BS_RPAD + kk);
#pragma unroll
            for (int q = 0; q < BS_CQ; ++q) {
              const int j = warp + BS_WARPS * q;
              if (j < ct) {                           // warp-uniform
                const float4 cv = *reinterpret_cast<const float4*>(cand_s + (size_t)j * H + k0 + kk);
                fma4(acc[0][q], r0, cv);
                fma4(acc[1][q], r1, cv);
              }
            }
          }
        }
        // max over this warp's candidate rows, then over the warps (fixed order)
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          float mx = -FLT_MAX;
#pragma unroll
          for (int q = 0; q < BS_CQ; ++q) {
            const int j = warp + BS_WARPS * q;
            if (j < ct) mx = fmaxf(mx, acc[m][q] * cinv_s[j]);
          }
          red_s[warp * BS_MT + lane + 32 * m] = mx;
        }
        __syncthreads();
        if (threadIdx.x < BS_MT) {
          float mx = best_s[threadIdx.x];
#pragma unroll
          for (int w = 0; w < BS_WARPS; ++w) mx = fmaxf(mx, red_s[w * BS_MT + threadIdx.x]);
          best_s[threadIdx.x] = mx;
        }
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        for (int m = 0; m < nt; ++m) {
          const int row = item_row[m], p = item_pair[m];
          run_sum += best_s[m] * a.inv_norm[row - a.row_begin];
          if (t0 + m == a.item_off[p + 1] - 1) {
            a.out[p] = run_sum / (float)(a.item_off[p + 1] - a.item_off[p]);
            run_sum = 0.f;
          }
        }
      }
    }
    __syncthreads();              // shared memory is reused by the next group
  }
}

size_t bs_smem_bytes(int H) {
  return sizeof(float) * ((size_t)BS_CT * H + BS_MT * BS_RPAD + BS_WARPS * BS_MT + BS_MT + BS_CT) +
         sizeof(int) * 2 * BS_MT;
}

}  // namespace

int launch_bertscore(const float* emb, const int32_t* row_off, const int32_t* pair_ref, const int32_t* item_off,
                     const int32_t* grp_pair, const int32_t* grp_cand, int32_t n_groups, int H, int32_t row_begin,
                     int32_t row_end, float* inv_norm, float* out, cudaStream_t s) {
  if (n_groups <= 0) return PLLB_OK;
  if (H % BS_KS != 0) return fail(PLLB_ERR_INVALID, "pllb_bertscore: hidden must be a multiple of 32");
  const size_t smem = bs_smem_bytes(H);
  // opt_in_smem runs once per kernel and device: opt in for the largest supported hidden size
  PLLB_CUDA(opt_in_smem(bertscore_recall_kernel, (int)bs_smem_bytes(1024)));
  int per_sm = 0;
  PLLB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bertscore_recall_kernel, BS_THREADS, smem));
  if (per_sm < 1) return fail(PLLB_ERR_INVALID, "pllb_bertscore: hidden size too large for shared memory");
  const int grid = per_sm * sm_count();       // co-resident: the grid sync needs every CTA on the device at once
  BsArgs args{emb, row_off, pair_ref, item_off, grp_pair, grp_cand, inv_norm, out, n_groups, H, row_begin, row_end};
  void* params[] = {&args};
  PLLB_CUDA(cudaLaunchCooperativeKernel((const void*)bertscore_recall_kernel, dim3(grid), dim3(BS_THREADS), params, smem, s));
  PLLB_LAUNCH_CHECK("bertscore_recall_kernel");
  return PLLB_OK;
}

}  // namespace pllb
