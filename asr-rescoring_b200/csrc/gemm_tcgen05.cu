// gemm_tcgen05.cu — the encoder / MLM-head GEMM for sm_100a.
//
//   C[M,N] = A[M,K] * W[N,K]^T  (+ fused epilogue)
//
// A (activations) and W (nn.Linear weight, [out,in]) are both K-contiguous bf16, so the
// "TN" form maps straight onto K-major UMMA operands with no transposes.  This replaces
// the six F.linear calls per BertLayer of transformers' modeling_bert.py:179-181,295,340,353
// and the MLM head's transform / decoder (:481-501) that MLM_PLL/main.py:89-94 invokes.
//
// Design (one CTA per SM, persistent over output tiles):
//   warp 0   : TMA producer — cp.async.bulk.tensor loads of a 128x64 A box and a 256x64 W
//              box (128-byte swizzle) into a 4-stage shared-memory ring, mbarrier-tracked.
//   warp 1   : MMA issuer — one thread issues tcgen05.mma (M=128, N=256, K=16) x4 per
//              stage; accumulators live in TMEM (2 x 256 fp32 columns, double buffered so
//              the epilogue of tile i overlaps the MMAs of tile i+1); tcgen05.commit frees
//              smem stages and publishes finished accumulators.
//   warps 2-9: epilogue (two warps per TMEM lane quarter, half of the tile's columns each)
//              — tcgen05.ld (32 lanes x 32 columns per warp), bias / erf-GELU /
//              dtype conversion in registers, 128-byte-swizzled staging in shared memory
//              and TMA stores; or, for the decoder, an online logsumexp over the vocab
//              tile plus the label-column pick, so the [copies x V] logits never exist; or, for
//              greedy generation, the tile's (max, first argmax) pair, with the same column pick; or,
//              for beam search, the logsumexp pair plus the tile's KSEL largest (logit, column) pairs.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <climits>

#include "common.h"
#include "ptx.cuh"

namespace pllb {

namespace {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
constexpr int STAGES = 4;
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BM * BK * 2;   // 16 KiB
constexpr int B_STAGE_BYTES = BN * BK * 2;   // 32 KiB
constexpr int EPI_WARPS = 8;                 // two per TMEM lane quarter, each owning half of the BN columns
constexpr int EPI_COLS = BN / 2;             // columns per epilogue warp
constexpr int EPI_BUF_BYTES = 32 * 128;      // one 32-row x 128-byte swizzled box
constexpr int EPI_BUFS = 1;                  // per epilogue warp
constexpr int NUM_THREADS = 32 * (2 + EPI_WARPS);
constexpr int TMEM_COLS = 512;               // 2 accumulator stages x BN columns
constexpr int SMEM_PIPE = STAGES * (A_STAGE_BYTES + B_STAGE_BYTES);
constexpr int SMEM_EPI = EPI_WARPS * EPI_BUFS * EPI_BUF_BYTES;
constexpr int SMEM_BARS = 256;
constexpr int SMEM_TOTAL = SMEM_PIPE + SMEM_EPI + SMEM_BARS + 1024;  // + alignment slack

struct KParams {
  int M, N, K;
  const float* bias;
  LseArgs lse;
};

// HF activations "gelu" = nn.functional.gelu (erf form): 0.5 x (1 + erf(x / sqrt 2)).
// With K = 768 the tensor core finishes a 128x256 tile in ~6 k cycles, which leaves the four
// SM sub-partitions ~24 issue slots per output element for the whole epilogue: erff()
// (~30 instructions) or any two-MUFU formula makes the epilogue, not the MMA, pace FFN1.
//
// fp32 output (MLM head transform, few rows): Abramowitz-Stegun 7.1.26, |err| <= 1.5e-7,
// with 1 + erf formed without cancellation on the negative side.
__device__ __forceinline__ float gelu_erf(float x) {
  const float z = fabsf(x) * 0.70710678118654752440f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float pe = p * t * __expf(-z * z);          // 1 - erf(|x| / sqrt 2)
  const float one_plus_erf = x >= 0.f ? 2.0f - pe : pe;
  return 0.5f * x * one_plus_erf;
}
// bf16 output (FFN1, every token): MUFU-free, two elements per instruction (FFMA2).
// erf(z) ~= z * P(z^2) on |z| <= 3 (degree-8 minimax fit, |err| <= 1.7e-5), +-1 beyond
// (1 - erf(3) = 2.2e-5): |gelu error| <= 6e-5 absolute for x < 0 and <= 3e-5 relative for
// x > 0 — an order of magnitude below the bf16 rounding (2^-9 relative) applied right after.
__device__ __forceinline__ float2 gelu_erf2(float2 x) {
  float2 z = fmul2(x, make_float2(0.70710678118654752440f, 0.70710678118654752440f));
  z.x = fminf(fmaxf(z.x, -3.0f), 3.0f);
  z.y = fminf(fmaxf(z.y, -3.0f), 3.0f);
  const float2 u = fmul2(z, z);
  float2 p = make_float2(4.074217013e-08f, 4.074217013e-08f);
  p = ffma2(p, u, make_float2(-1.944825010e-06f, -1.944825010e-06f));
  p = ffma2(p, u, make_float2(4.106055743e-05f, 4.106055743e-05f));
  p = ffma2(p, u, make_float2(-5.110371206e-04f, -5.110371206e-04f));
  p = ffma2(p, u, make_float2(4.235428517e-03f, 4.235428517e-03f));
  p = ffma2(p, u, make_float2(-2.510286391e-02f, -2.510286391e-02f));
  p = ffma2(p, u, make_float2(1.110793386e-01f, 1.110793386e-01f));
  p = ffma2(p, u, make_float2(-3.753148772e-01f, -3.753148772e-01f));
  p = ffma2(p, u, make_float2(1.128268426e+00f, 1.128268426e+00f));
  const float2 e = fmul2(p, z);
  const float2 hx = fmul2(x, make_float2(0.5f, 0.5f));
  return ffma2(hx, e, hx);
}

// two fp32 -> one packed 16-bit pair in the operand dtype of the handle (bf16 or fp16)
template <bool FP16>
__device__ __forceinline__ uint32_t pack16x2(float lo, float hi) {
  return pack16x2_sat<FP16>(lo, hi);
}

// MC: the kernel runs as clusters of two CTAs that work on vertically adjacent tiles (same
// weight columns): each CTA fetches half of the 256x64 W box and TMA-multicasts it to both,
// which halves the L2 -> SM weight traffic; the stage-release barrier then counts both CTAs.
//
// MODE 2 (cta_group::2): the pair issues ONE tcgen05.mma with M = 256 per k-step from the leader
// CTA; each CTA keeps its own 128 rows of A and only HALF of the W box (the tensor cores read
// the other half from the peer's shared memory), so a stage is 32 KiB instead of 48 and the
// ring is 6 deep; accumulators for rows 0-127 / 128-255 land in the leader's / peer's TMEM.
// Both CTAs' TMA loads complete on the leader's full barrier; the MMA's commits are multicast
// to both CTAs (stage release, accumulator ready); both epilogues report back to the leader.
template <int EPI, int DT, int MODE>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, const KParams p) {
  constexpr bool MC = MODE == 1;
  constexpr bool TWO = MODE == 2;
  constexpr bool FP16 = (DT & 4) != 0;          // type of the 16-bit output
  // TWO: 5 x 32 KiB operand stages + two staging boxes per epilogue warp; else 4 x 48 KiB + one box
  constexpr int NST = TWO ? 5 : STAGES;
  constexpr int B_BYTES = TWO ? B_STAGE_BYTES / 2 : B_STAGE_BYTES;
  constexpr int EBUFS = TWO ? 2 : EPI_BUFS;
  constexpr int PIPE_BYTES = NST * (A_STAGE_BYTES + B_BYTES);
  static_assert(PIPE_BYTES + EPI_WARPS * EBUFS * EPI_BUF_BYTES <= SMEM_PIPE + SMEM_EPI, "shared memory budget");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + NST * A_STAGE_BYTES;
  const uint32_t sEpi = smem_base + PIPE_BYTES;
  const uint32_t sBar = smem_base + SMEM_PIPE + SMEM_EPI;
  const uint32_t bar_full = sBar;                 // NST x 8 B
  const uint32_t bar_empty = sBar + 8 * NST;      // NST x 8 B
  const uint32_t bar_tfull = sBar + 16 * NST;     // 2 x 8 B
  const uint32_t bar_tempty = bar_tfull + 16;     // 2 x 8 B
  const uint32_t tmem_slot = bar_tempty + 16;     // 4 B
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int tiles_n = p.N / BN;
  const int tiles_m = (p.M + BM - 1) / BM;
  const int num_kb = p.K / BK;
  // work units: one tile per CTA, or (MC) a pair of vertically adjacent tiles per cluster
  constexpr bool PAIR = MC || TWO;
  const uint32_t crank = PAIR ? cluster_ctarank() : 0;
  const int unit0 = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int unit_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const int num_tiles = (PAIR ? (tiles_m + 1) / 2 : tiles_m) * tiles_n;
#define PLLB_TILE_M(tile) ((PAIR ? 2 * ((tile) / tiles_n) + (int)crank : (tile) / tiles_n) * BM)

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
    if (EPI != EPI_LSE && EPI != EPI_ARGMAX && EPI != EPI_TOPK8 && EPI != EPI_TOPK16) prefetch_tensormap(&tmC);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < NST; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, MC ? 2 : 1);           // MC: both CTAs' MMAs must have retired
      }
      for (int s = 0; s < 2; ++s) {
        mbar_init(bar_tfull + 8 * s, 1);
        mbar_init(bar_tempty + 8 * s, TWO ? 2 * EPI_WARPS : EPI_WARPS);   // TWO: both CTAs' epilogues
      }
      fence_barrier_init();
    }
    __syncwarp();
    if constexpr (TWO) {
      tmem_alloc_2cta(tmem_slot, TMEM_COLS);
      tmem_relinquish_2cta();
    } else {
      tmem_alloc(tmem_slot, TMEM_COLS);
      tmem_relinquish();
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();     // the peer's barriers exist before anything is multicast to them
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int tile = unit0; tile < num_tiles; tile += unit_stride) {
        const int m0 = PLLB_TILE_M(tile);
        const int n0 = (tile % tiles_n) * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1);
          if constexpr (TWO) {
            // both CTAs' bytes are counted on the leader's barrier, which only the leader arms
            const uint32_t lead_full = mapa_shared(bar_full + 8 * stage, 0);
            if (crank == 0) mbar_arrive_expect_tx(bar_full + 8 * stage, 2 * (A_STAGE_BYTES + B_BYTES));
            tma_load_2d_2sm(sA + stage * A_STAGE_BYTES, &tmA, lead_full, kb * BK, m0);
            tma_load_2d_2sm(sB + stage * B_BYTES, &tmB, lead_full, kb * BK, n0 + (int)crank * (BN / 2));
            if (++stage == NST) { stage = 0; phase ^= 1; }
            continue;
          }
          mbar_arrive_expect_tx(bar_full + 8 * stage, A_STAGE_BYTES + B_STAGE_BYTES);
          tma_load_2d(sA + stage * A_STAGE_BYTES, &tmA, bar_full + 8 * stage, kb * BK, m0);
          if constexpr (MC) {
            // my half of the W box (128 rows = 16 KiB), delivered to both CTAs
            tma_load_2d_multicast(sB + stage * B_STAGE_BYTES + crank * (B_STAGE_BYTES / 2), &tmB, bar_full + 8 * stage,
                                  kb * BK, n0 + (int)crank * (BN / 2), (uint16_t)0x3);
          } else
          tma_load_2d(sB + stage * B_STAGE_BYTES, &tmB, bar_full + 8 * stage, kb * BK, n0);
          if (++stage == NST) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------ MMA issuer
    if (lane == 0 && (!TWO || crank == 0)) {                 // TWO: the leader issues for the pair
      constexpr int MMA_M = TWO ? 2 * BM : BM;
      constexpr uint32_t idesc = make_idesc_16(MMA_M, BN, (DT & 1) != 0, (DT & 2) != 0);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int tile = unit0; tile < num_tiles; tile += unit_stride) {
        mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);   // epilogue drained this accumulator
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(bar_full + 8 * stage, phase);         // TMA bytes landed
          tcgen05_fence_after();
          const uint32_t a_addr = sA + stage * A_STAGE_BYTES;
          const uint32_t b_addr = sB + stage * B_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            const uint64_t adesc = make_kmajor_sw128_desc(a_addr + k * UMMA_K * 2);
            const uint64_t bdesc = make_kmajor_sw128_desc(b_addr + k * UMMA_K * 2);
            if constexpr (TWO) tcgen05_mma_bf16_2cta(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
            else tcgen05_mma_bf16(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          // smem stage reusable once the MMAs retire (in every CTA that holds a part of it)
          if constexpr (TWO) tcgen05_commit_2cta_multicast(bar_empty + 8 * stage, (uint16_t)0x3);
          else if constexpr (MC) tcgen05_commit_multicast(bar_empty + 8 * stage, (uint16_t)0x3);
          else tcgen05_commit(bar_empty + 8 * stage);
          if (++stage == NST) { stage = 0; phase ^= 1; }
        }
        // accumulator complete (TWO: both CTAs' epilogues read their own 128 rows)
        if constexpr (TWO) tcgen05_commit_2cta_multicast(bar_tfull + 8 * acc, (uint16_t)0x3);
        else tcgen05_commit(bar_tfull + 8 * acc);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // ------------------------------------------------------------ epilogue warps
    const int q = warp & 3;                               // TMEM lane quarter this warp may read
    const int ew = warp - 2;
    const int cbase = (ew >> 2) * EPI_COLS;               // first tile column owned by this warp
    const uint32_t my_buf = sEpi + ew * EBUFS * EPI_BUF_BYTES;
    uint32_t acc = 0, acc_phase = 0, buf_i = 0;
    // The accumulator buffer goes back to the MMA warp as soon as its last columns sit in registers
    // (16-bit epilogues: before the bias / GELU math and the stores of the last 64 columns), not after them.
    auto release_acc = [&]() {
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (TWO) mbar_arrive_cluster(mapa_shared(bar_tempty + 8 * acc, 0));   // the leader's MMA waits for both
        else mbar_arrive(bar_tempty + 8 * acc);
      }
    };
    for (int tile = unit0; tile < num_tiles; tile += unit_stride) {
      const int m0 = PLLB_TILE_M(tile);
      const int tn = tile % tiles_n;
      const int n0 = tn * BN;
      const int row = m0 + q * 32 + lane;
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tcgen05_fence_after();
      const uint32_t t_addr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16);

      if constexpr (EPI == EPI_LSE) {
        const int label = (row < p.M) ? p.lse.labels[row] : -1;
        float run_max = -INFINITY, run_sum = 0.f, lab_val = 0.f;
        bool has_label = false;
        for (int c0 = cbase; c0 < cbase + EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_addr + c0, r);
          tcgen05_wait_ld();
          float x[32];
          float cmax = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = n0 + c0 + j;
            float v = __uint_as_float(r[j]) + __ldg(p.bias + col);
            if (col >= p.lse.vocab) v = -INFINITY;
            if (col == label) { lab_val = v; has_label = true; }
            x[j] = v;
            cmax = fmaxf(cmax, v);
          }
          if (cmax > -INFINITY) {
            const float new_max = fmaxf(run_max, cmax);
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) s += __expf(x[j] - new_max);
            run_sum = run_sum * __expf(run_max - new_max) + s;
            run_max = new_max;
          }
        }
        if (row < p.M) {
          p.lse.partials[((size_t)row * tiles_n + tn) * 2 + (ew >> 2)] = make_float2(run_max, run_sum);
          if (has_label) p.lse.label_logit[row] = lab_val;
        }
      } else if constexpr (EPI == EPI_ARGMAX) {
        // greedy decoding: (max, first column attaining it) of this half tile; columns ascend and the
        // comparison is strict, so a tie keeps the lower column, as torch.argmax does
        const int label = (row < p.M) ? p.lse.labels[row] : -1;
        float run_max = -INFINITY, lab_val = 0.f;
        int run_arg = n0 + cbase;
        bool has_label = false;
        for (int c0 = cbase; c0 < cbase + EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_addr + c0, r);
          tcgen05_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = n0 + c0 + j;
            float v = __uint_as_float(r[j]) + __ldg(p.bias + col);
            if (col >= p.lse.vocab) v = -INFINITY;
            if (col == label) { lab_val = v; has_label = true; }
            if (v > run_max) { run_max = v; run_arg = col; }
          }
        }
        if (row < p.M) {
          p.lse.partials[((size_t)row * tiles_n + tn) * 2 + (ew >> 2)] = make_float2(run_max, __int_as_float(run_arg));
          if (has_label) p.lse.label_logit[row] = lab_val;
        }
      } else if constexpr (EPI == EPI_TOPK8 || EPI == EPI_TOPK16) {
        // beam search: the (max, sum of exp) pair exactly as EPI_LSE, plus the KS largest (logit, column)
        // pairs of this half tile in descending order, ties to the lower column.  The list starts as
        // (-inf, INT_MAX) placeholders, so masked columns (-inf) still fill it by ascending column.
        constexpr int KS = EPI == EPI_TOPK16 ? 16 : 8;
        float run_max = -INFINITY, run_sum = 0.f;
        float tv[KS];
        int tc[KS];
#pragma unroll
        for (int i = 0; i < KS; ++i) { tv[i] = -INFINITY; tc[i] = INT_MAX; }
        for (int c0 = cbase; c0 < cbase + EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_addr + c0, r);
          tcgen05_wait_ld();
          float x[32];
          float cmax = -INFINITY;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = n0 + c0 + j;
            float v = __uint_as_float(r[j]) + __ldg(p.bias + col);
            if (col >= p.lse.vocab) v = -INFINITY;
            x[j] = v;
            cmax = fmaxf(cmax, v);
          }
          if (cmax > -INFINITY) {
            const float new_max = fmaxf(run_max, cmax);
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) s += __expf(x[j] - new_max);
            run_sum = run_sum * __expf(run_max - new_max) + s;
            run_max = new_max;
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            // columns ascend: a value equal to the last kept one enters only in front of a placeholder
            if (x[j] > tv[KS - 1] || (x[j] == tv[KS - 1] && tc[KS - 1] == INT_MAX)) {
              tv[KS - 1] = x[j];
              tc[KS - 1] = n0 + c0 + j;
#pragma unroll
              for (int i = KS - 1; i > 0; --i) {
                if (tv[i] > tv[i - 1] || (tv[i] == tv[i - 1] && tc[i] < tc[i - 1])) {
                  const float fv = tv[i]; tv[i] = tv[i - 1]; tv[i - 1] = fv;
                  const int fc = tc[i]; tc[i] = tc[i - 1]; tc[i - 1] = fc;
                }
              }
            }
          }
        }
        if (row < p.M) {
          const size_t slot = ((size_t)row * tiles_n + tn) * 2 + (ew >> 2);
          p.lse.partials[slot] = make_float2(run_max, run_sum);
          // the top-KS lists follow the [M, 2 * tiles_n] pairs: [M, 2 * tiles_n, KS] (logit, column)
          float4* top = reinterpret_cast<float4*>(p.lse.partials + (size_t)p.M * tiles_n * 2 + slot * KS);
#pragma unroll
          for (int i = 0; i < KS; i += 2)
            top[i / 2] = make_float4(tv[i], __int_as_float(tc[i]), tv[i + 1], __int_as_float(tc[i + 1]));
        }
      } else if constexpr (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_BF16) {
        for (int c0 = cbase; c0 < cbase + EPI_COLS; c0 += 64) {
          uint32_t r0[32], r1[32];
          tmem_ld_32x32b_x32(t_addr + c0, r0);
          tmem_ld_32x32b_x32(t_addr + c0 + 32, r1);
          tcgen05_wait_ld();
          if (c0 + 64 >= cbase + EPI_COLS) release_acc();   // last columns are in registers
          const uint32_t buf = my_buf + (buf_i % EBUFS) * EPI_BUF_BYTES;
          if (lane == 0) tma_store_wait_read<EBUFS - 1>();      // the store that last read this buffer is done
          __syncwarp();
          ++buf_i;
          const float4* bias4 = reinterpret_cast<const float4*>(p.bias + n0 + c0);
#pragma unroll
          for (int c = 0; c < 8; ++c) {                    // 8 chunks of 8 bf16 (16 B)
            float2 v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int cc = c * 8 + 2 * j;
              v[j] = make_float2(__uint_as_float(cc < 32 ? r0[cc] : r1[cc - 32]),
                                 __uint_as_float(cc < 32 ? r0[cc + 1] : r1[cc - 31]));
            }
            const float4 b0 = __ldg(bias4 + 2 * c), b1 = __ldg(bias4 + 2 * c + 1);
            v[0] = fadd2(v[0], make_float2(b0.x, b0.y));
            v[1] = fadd2(v[1], make_float2(b0.z, b0.w));
            v[2] = fadd2(v[2], make_float2(b1.x, b1.y));
            v[3] = fadd2(v[3], make_float2(b1.z, b1.w));
            if constexpr (EPI == EPI_BIAS_GELU_BF16) {
#pragma unroll
              for (int j = 0; j < 4; ++j) v[j] = gelu_erf2(v[j]);
            }
            const uint32_t dst = buf + lane * 128 + ((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pack16x2<FP16>(v[0].x, v[0].y)),
                         "r"(pack16x2<FP16>(v[1].x, v[1].y)), "r"(pack16x2<FP16>(v[2].x, v[2].y)),
                         "r"(pack16x2<FP16>(v[3].x, v[3].y))
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmC, buf, n0 + c0, m0 + q * 32);
            tma_store_commit();
          }
        }
      } else {  // fp32 output
        for (int c0 = cbase; c0 < cbase + EPI_COLS; c0 += 32) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(t_addr + c0, r);
          tcgen05_wait_ld();
          const uint32_t buf = my_buf + (buf_i % EBUFS) * EPI_BUF_BYTES;
          if (lane == 0) tma_store_wait_read<EBUFS - 1>();
          __syncwarp();
          ++buf_i;
          const float4* bias4 = reinterpret_cast<const float4*>(p.bias + n0 + c0);
#pragma unroll
          for (int c = 0; c < 8; ++c) {                    // 8 chunks of 4 fp32 (16 B)
            const float4 b = __ldg(bias4 + c);
            float v0 = __uint_as_float(r[4 * c + 0]) + b.x;
            float v1 = __uint_as_float(r[4 * c + 1]) + b.y;
            float v2 = __uint_as_float(r[4 * c + 2]) + b.z;
            float v3 = __uint_as_float(r[4 * c + 3]) + b.w;
            if constexpr (EPI == EPI_BIAS_GELU_F32) {
              v0 = gelu_erf(v0); v1 = gelu_erf(v1); v2 = gelu_erf(v2); v3 = gelu_erf(v3);
            }
            const uint32_t dst = buf + lane * 128 + ((c ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(__float_as_uint(v0)),
                         "r"(__float_as_uint(v1)), "r"(__float_as_uint(v2)), "r"(__float_as_uint(v3))
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmC, buf, n0 + c0, m0 + q * 32);
            tma_store_commit();
          }
        }
      }
      // all tcgen05.ld of this accumulator have completed (wait::ld above): release it
      if constexpr (EPI != EPI_BIAS_BF16 && EPI != EPI_BIAS_GELU_BF16) release_acc();
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    if (lane == 0) tma_store_wait_all();
  }

  tcgen05_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();     // the peer may still multicast-arrive on this CTA's barriers
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    if constexpr (TWO) tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
#undef PLLB_TILE_M
}

// ------------------------------------------------------------------ host side
int make_tmap(CUtensorMap* m, const void* base, CUtensorMapDataType dt, int elt_bytes, uint64_t rows, uint64_t cols,
              uint32_t box_rows, uint32_t box_cols) {
  return get_tmap_2d(m, base, dt, elt_bytes, rows, cols, box_rows, box_cols);
}

template <int EPI, int DT, int MODE>
int launch_epi3(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, const KParams& kp, int grid,
                cudaStream_t stream) {
  auto kern = gemm_tcgen05_kernel<EPI, DT, MODE>;
  PLLB_CUDA(opt_in_smem(kern, SMEM_TOTAL));
  if constexpr (MODE != 0) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = SMEM_TOTAL;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    PLLB_CUDA(cudaLaunchKernelEx(&cfg, kern, a, b, c, kp));
    ++g_launch_counter;
  } else {
    kern<<<grid, NUM_THREADS, SMEM_TOTAL, stream>>>(a, b, c, kp);
    PLLB_LAUNCH_CHECK("gemm_tcgen05_kernel");
  }
  return PLLB_OK;
}
template <int EPI, int DT>
int launch_epi2(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, const KParams& kp, int grid, int mode,
                cudaStream_t stream) {
  if (mode == 2) return launch_epi3<EPI, DT, 2>(a, b, c, kp, grid, stream);
  if (mode == 1) return launch_epi3<EPI, DT, 1>(a, b, c, kp, grid, stream);
  return launch_epi3<EPI, DT, 0>(a, b, c, kp, grid, stream);
}
template <int EPI>
int launch_epi(const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, const KParams& kp, int grid, int dt,
               int mode, cudaStream_t stream) {
  switch (dt) {
    case DT_BF16: return launch_epi2<EPI, DT_BF16>(a, b, c, kp, grid, mode, stream);
    case DT_FP16: return launch_epi2<EPI, DT_FP16>(a, b, c, kp, grid, mode, stream);
  }
  return fail(PLLB_ERR_INVALID, "gemm: unsupported operand dtype combination");
}

// 0 = one CTA per tile, 1 = CTA pairs with TMA multicast of W, 2 = cta_group::2 MMA.
// M > 128: cta_group::2, except for the GELU epilogue — FFN1 is paced by its epilogue's CUDA-core
// math, where the cluster-scope accumulator hand-back of mode 2 costs more than the deeper
// operand ring gains (measured ABAB inside the C2 step: QKV 671 vs 727 ms, FFN1 905-918 vs 884 ms).
int pair_mode(int epilogue) { return epilogue == EPI_BIAS_GELU_BF16 ? 1 : 2; }

}  // namespace

int launch_gemm_tcgen05(const void* A, const void* W, const float* bias, void* C, int64_t M, int N, int K,
                        int epilogue, const LseArgs* lse, int dt, cudaStream_t stream) {
  if (M <= 0) return PLLB_OK;
  if (N % BN != 0 || K % BK != 0 || M > INT32_MAX)
    return fail(PLLB_ERR_INVALID, "gemm: need N % 256 == 0 and K % 64 == 0");
  CUtensorMap ta, tb, tc;
  int rc;
  if ((rc = make_tmap(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)M, (uint64_t)K, BM, BK))) return rc;
  const int mode = M > BM ? pair_mode(epilogue) : 0;             // pairs of vertically adjacent tiles share W
  const bool mc = mode != 0;
  if ((rc = make_tmap(&tb, W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)N, (uint64_t)K, mc ? BN / 2 : BN, BK))) return rc;
  tc = ta;
  if (epilogue == EPI_BIAS_BF16 || epilogue == EPI_BIAS_GELU_BF16) {
    if ((rc = make_tmap(&tc, C, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)M, (uint64_t)N, 32, 64))) return rc;
  } else if (epilogue == EPI_BIAS_F32 || epilogue == EPI_BIAS_GELU_F32) {
    if ((rc = make_tmap(&tc, C, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (uint64_t)M, (uint64_t)N, 32, 32))) return rc;
  }
  KParams kp{};
  kp.M = (int)M; kp.N = N; kp.K = K; kp.bias = bias;
  if (epilogue == EPI_LSE || epilogue == EPI_ARGMAX || epilogue == EPI_TOPK8 || epilogue == EPI_TOPK16) {
    if (!lse) return fail(PLLB_ERR_INVALID, "gemm: LSE / argmax / top-k epilogue needs LseArgs");
    kp.lse = *lse;
  }
  int grid;
  const int sms = sm_count();
  if (mc) {
    const int64_t units = ceil_div(ceil_div(M, BM), 2) * (N / BN);
    const int64_t clusters = units < sms / 2 ? units : sms / 2;
    grid = (int)(2 * clusters);
  } else {
    const int64_t tiles = ceil_div(M, BM) * (N / BN);
    grid = (int)(tiles < sms ? tiles : sms);
  }
  switch (epilogue) {
    case EPI_BIAS_BF16: return launch_epi<EPI_BIAS_BF16>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_BIAS_GELU_BF16: return launch_epi<EPI_BIAS_GELU_BF16>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_BIAS_F32: return launch_epi<EPI_BIAS_F32>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_BIAS_GELU_F32: return launch_epi<EPI_BIAS_GELU_F32>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_LSE: return launch_epi<EPI_LSE>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_ARGMAX: return launch_epi<EPI_ARGMAX>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_TOPK8: return launch_epi<EPI_TOPK8>(ta, tb, tc, kp, grid, dt, mode, stream);
    case EPI_TOPK16: return launch_epi<EPI_TOPK16>(ta, tb, tc, kp, grid, dt, mode, stream);
  }
  return fail(PLLB_ERR_INVALID, "gemm: unknown epilogue");
}

// ------------------------------------------------------------------ SIMT validation kernel
// Plain shared-memory-tiled GEMM with the same operand rounding and epilogues; used by
// tests to localise errors of the tcgen05 path (never on the timed path).
namespace {
template <int EPI>
__global__ void gemm_simt_kernel(const __nv_bfloat16* __restrict__ A, const __nv_bfloat16* __restrict__ W,
                                 const float* __restrict__ bias, void* __restrict__ C, int M, int N, int K) {
  __shared__ float As[16][17], Ws[16][17];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const int row = blockIdx.y * 16 + ty, col = blockIdx.x * 16 + tx;
  float acc = 0.f;
  for (int k0 = 0; k0 < K; k0 += 16) {
    As[ty][tx] = (row < M) ? __bfloat162float(A[(size_t)row * K + k0 + tx]) : 0.f;
    const int wrow = blockIdx.x * 16 + ty;
    Ws[ty][tx] = (wrow < N) ? __bfloat162float(W[(size_t)wrow * K + k0 + tx]) : 0.f;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) acc += As[ty][k] * Ws[tx][k];
    __syncthreads();
  }
  if (row < M && col < N) {
    float v = acc + bias[col];
    if (EPI == EPI_BIAS_GELU_BF16 || EPI == EPI_BIAS_GELU_F32) v = gelu_erf(v);
    if (EPI == EPI_BIAS_BF16 || EPI == EPI_BIAS_GELU_BF16)
      reinterpret_cast<__nv_bfloat16*>(C)[(size_t)row * N + col] = __float2bfloat16_rn(v);
    else
      reinterpret_cast<float*>(C)[(size_t)row * N + col] = v;
  }
}
}  // namespace

int launch_gemm_simt(const void* A, const void* W, const float* bias, void* C, int64_t M, int N, int K, int epilogue,
                     cudaStream_t stream) {
  if (M <= 0) return PLLB_OK;
  if (K % 16 != 0) return fail(PLLB_ERR_INVALID, "gemm_simt: K % 16 != 0");
  dim3 block(16, 16), grid((unsigned)ceil_div(N, 16), (unsigned)ceil_div(M, 16));
  const __nv_bfloat16* a = reinterpret_cast<const __nv_bfloat16*>(A);
  const __nv_bfloat16* w = reinterpret_cast<const __nv_bfloat16*>(W);
  switch (epilogue) {
    case EPI_BIAS_BF16: gemm_simt_kernel<EPI_BIAS_BF16><<<grid, block, 0, stream>>>(a, w, bias, C, (int)M, N, K); break;
    case EPI_BIAS_GELU_BF16: gemm_simt_kernel<EPI_BIAS_GELU_BF16><<<grid, block, 0, stream>>>(a, w, bias, C, (int)M, N, K); break;
    case EPI_BIAS_F32: gemm_simt_kernel<EPI_BIAS_F32><<<grid, block, 0, stream>>>(a, w, bias, C, (int)M, N, K); break;
    case EPI_BIAS_GELU_F32: gemm_simt_kernel<EPI_BIAS_GELU_F32><<<grid, block, 0, stream>>>(a, w, bias, C, (int)M, N, K); break;
    default: return fail(PLLB_ERR_INVALID, "gemm_simt: unsupported epilogue");
  }
  PLLB_LAUNCH_CHECK("gemm_simt_kernel");
  return PLLB_OK;
}

}  // namespace pllb
