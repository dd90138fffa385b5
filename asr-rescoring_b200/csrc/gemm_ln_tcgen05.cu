// gemm_ln_tcgen05.cu — GEMM with the bias + residual + LayerNorm epilogue fused in:
//
//   hidden = LayerNorm(A[M,K] * W[H,K]^T + bias + hidden)          (in place, fp32)
//   hidden16 = bf16/fp16(hidden)                                    (operand of the next GEMM)
//
// i.e. BertSelfOutput / BertOutput (transformers modeling_bert.py:294-298, 352-356) in one
// kernel.  The separate LayerNorm kernel moves 10.5 KB per row and layer-half through HBM
// (pre-LN fp32 out and back in, residual in, fp32 + 16-bit out); fused, the residual is
// read once and the two outputs written once (7.5 KB), and the 3 KB pre-LN round trip
// disappears.
//
// A LayerNorm row spans H = 768 / 1024 columns, more than the 512 fp32 TMEM columns one SM
// owns, so a thread-block CLUSTER of CN = H/256 CTAs covers one 128-row block: CTA rank r
// computes the 128x256 tile of columns [256r, 256r+256) with the same TMA -> tcgen05.mma ->
// TMEM pipeline as gemm_tcgen05.cu; its epilogue warps pull the tile into registers (one row
// per thread, 128 columns each), add bias and the residual (read straight from the T32
// blocked fp32 layout, fully coalesced), reduce (mean, M2) per row inside the CTA, exchange the per-CTA pair with
// the peer CTAs through distributed shared memory (st.shared::cluster + a cluster-scope
// mbarrier), merge them with Chan's formula, normalise from registers, write the fp32 stream
// back in place and TMA-store the 16-bit operand copy.  No second pass over TMEM or HBM.
#include <cooperative_groups.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>

#include "common.h"
#include "ptx.cuh"

namespace pllb {

namespace {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;
// STAGED = true : 3-stage operand ring + the 16-bit output through two swizzled boxes per warp and TMA
//                 stores (best when the epilogue paces the kernel: K = H, attention output);
// STAGED = false: 4-stage operand ring, 16-bit output written straight from registers (best when
//                 the mainloop paces the kernel: K = 4H, FFN2).
constexpr int UMMA_K = 16;
constexpr int A_STAGE_BYTES = BM * BK * 2;
constexpr int B_STAGE_BYTES = BN * BK * 2;
constexpr int EPI_WARPS = 8;
constexpr int EPI_COLS = BN / 2;               // columns per epilogue thread
constexpr int BOX_BYTES = 32 * 128;            // 32 rows x 128 B swizzled box
constexpr int NUM_THREADS = 32 * (2 + EPI_WARPS);
constexpr int TMEM_COLS = 512;
constexpr int MAX_CN = 4;

template <int CN>
constexpr int smem_xchg() { return 2 * 2 * CN * BM * 8; }                 // [parity][rank*2+half][row] float2
constexpr int SMEM_BARS = 512;
constexpr int SMEM_LIMIT = 232448;             // 227 KiB of dynamic shared memory per CTA
// bias | gamma | beta of this CTA's 256 columns, staged once.  The epilogue reads 12 float4 of them per
// 16-column chunk on its dependent chain; as global loads they compete for the ~28 KB of L1 that
// 227 KB of shared memory leave with the residual stream passing through (131 KB per tile), so a
// good part of them are L2 round trips.  From shared memory they cost one fixed short latency.
constexpr int SMEM_PAR = 3 * BN * 4;
template <bool STAGED, bool PAIR>
constexpr int ln_stages() {
  return PAIR ? (STAGED ? 4 : 6) : (STAGED ? 3 : 4);
}
template <int CN, bool STAGED, bool PAIR>
constexpr int smem_without_params() {
  return ln_stages<STAGED, PAIR>() * (A_STAGE_BYTES + (PAIR ? B_STAGE_BYTES / 2 : B_STAGE_BYTES)) +
         (STAGED ? EPI_WARPS * 2 * BOX_BYTES : 0) + smem_xchg<CN>() + SMEM_BARS + 1024;
}
// (the staged single-CTA form at H = 1024 has no 3 KB left: it keeps the global loads)
template <int CN, bool STAGED, bool PAIR>
constexpr bool params_in_smem() {
  return smem_without_params<CN, STAGED, PAIR>() + SMEM_PAR <= SMEM_LIMIT;
}
template <int CN, bool STAGED, bool PAIR>
constexpr int smem_total() {
  return smem_without_params<CN, STAGED, PAIR>() + (params_in_smem<CN, STAGED, PAIR>() ? SMEM_PAR : 0);
}

static_assert(smem_total<4, true, false>() <= SMEM_LIMIT && smem_total<4, false, false>() <= SMEM_LIMIT &&
              smem_total<4, true, true>() <= SMEM_LIMIT && smem_total<4, false, true>() <= SMEM_LIMIT &&
              smem_total<3, true, false>() <= SMEM_LIMIT, "shared memory budget of one CTA");

struct LnParams {
  int M, K, H;
  float* hidden;          // fp32 residual stream, T32 blocked layout, updated in place
  __nv_bfloat16* hidden16; // row-major 16-bit copy (bf16 or fp16 bits)
  const float* bias;
  const float* gamma;
  const float* beta;
  float eps;
};

template <bool FP16>
__device__ __forceinline__ uint32_t pack16x2(float lo, float hi) {
  return pack16x2_sat<FP16>(lo, hi);
}

__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t num_clusters_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa(uint32_t local_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
  return r;
}
// DSMEM message: 8-byte store into a peer CTA's shared memory that completes 8 tx bytes on the
// peer's mbarrier (SASS STAS) — no fences, no release/acquire round trips.
__device__ __forceinline__ void st_async_f32x2(uint32_t cluster_addr, float a, float b, uint32_t cluster_mbar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];"
               ::"r"(cluster_addr), "f"(a), "f"(b), "r"(cluster_mbar) : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 "
      "[%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tcgen05_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// ordered (volatile) loads: keeps ptxas from hoisting a tile's worth of parameter loads above
// the 128-register row slice and spilling it
__device__ __forceinline__ float4 ldg_f4_ordered(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
// PAIR: the cluster holds 2*CN CTAs and covers a 256-row block.  CTAs 2c and 2c+1 form a
// cta_group::2 pair on column group c: the leader issues ONE tcgen05.mma with M = 256 per k-step,
// each CTA stages its own 128 rows of A and only HALF of the 256 x 64 W box (a stage is 32 KiB
// instead of 48, the ring 6 / 4 deep instead of 4 / 3).  A single-CTA 128x256x16 MMA reads 12 KB
// of operands from shared memory per 128 tensor cycles while TMA writes the next stage — the
// shared-memory port, not the tensor pipe, paces that form (tensor pipe 63-67 % active in ncu);
// the pair reads 8 KB per CTA.  LayerNorm statistics are exchanged between the CN CTAs that hold
// the same rows (ranks rh, 2 + rh, 4 + rh).
template <int CN, int DT, bool STAGED, bool PAIR>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_ln_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmH16, const LnParams p) {
  constexpr bool FP16 = (DT & 4) != 0;          // type of the 16-bit output copy
  constexpr int STAGES = ln_stages<STAGED, PAIR>();
  constexpr int B_BYTES = PAIR ? B_STAGE_BYTES / 2 : B_STAGE_BYTES;
  constexpr int SMEM_PIPE = STAGES * (A_STAGE_BYTES + B_BYTES);
  constexpr int SMEM_EPI = STAGED ? EPI_WARPS * 2 * BOX_BYTES : 0;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - raw_addr);            // generic pointer to the aligned base
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + STAGES * A_STAGE_BYTES;
  const uint32_t sEpi = smem_base + SMEM_PIPE;
  const uint32_t sXchg = sEpi + SMEM_EPI;
  constexpr int SMEM_XCHG = smem_xchg<CN>();
  constexpr bool PAR_SMEM = params_in_smem<CN, STAGED, PAIR>();
  const uint32_t sBar = sXchg + SMEM_XCHG + (PAR_SMEM ? SMEM_PAR : 0);
  float* par_f = reinterpret_cast<float*>(smem_gen + SMEM_PIPE + SMEM_EPI + SMEM_XCHG);      // bias[256] | gamma[256] | beta[256]
  const float4* par4 = reinterpret_cast<const float4*>(par_f);
  float2* xchg = reinterpret_cast<float2*>(smem_gen + SMEM_PIPE + SMEM_EPI);   // [parity][rank*2+half][row]
  const uint32_t bar_full = sBar;                         // STAGES
  const uint32_t bar_empty = bar_full + 8 * STAGES;       // STAGES
  const uint32_t bar_tfull = bar_empty + 8 * STAGES;      // 2
  const uint32_t bar_tempty = bar_tfull + 16;             // 2
  const uint32_t bar_x = bar_tempty + 16;                 // 2 (cluster exchange, per parity)
  const uint32_t bar_r = bar_x + 16;                      // EPI_WARPS x 2 (residual boxes)
  const uint32_t tmem_slot = bar_r + 8 * EPI_WARPS * 2;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_gen + (tmem_slot - smem_base));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr bool CLUSTERED = CN > 1 || PAIR;
  const uint32_t rank = CLUSTERED ? cluster_ctarank() : 0;
  const uint32_t cg = PAIR ? rank >> 1 : rank;             // column group: columns [256 cg, 256 cg + 256)
  const uint32_t rh = PAIR ? rank & 1u : 0u;               // row half inside the 256-row block; 0 = leader of the pair
  const uint32_t leader = rank & ~1u;
  constexpr int ROWS = PAIR ? 2 * BM : BM;                 // rows of a block per cluster
  const int cluster = CLUSTERED ? (int)cluster_id_x() : (int)blockIdx.x;
  const int n_clusters = CLUSTERED ? (int)num_clusters_x() : (int)gridDim.x;
  const int tiles_m = (p.M + ROWS - 1) / ROWS;
  const int num_kb = p.K / BK;
  const int n0 = (int)cg * BN;
  // All CN CTAs of a cluster multiply the SAME 128 x K block of A by their own 256 columns of W.
  // With AMC the A stage (four 32-row boxes) is fetched from L2 once per cluster: CTA r issues
  // boxes r, r+CN, ... as TMA multicasts into every CTA's stage, and a stage is reused only after
  // every CTA's MMAs released it (their commits are multicast to all empty barriers).
  constexpr bool AMC = !PAIR && CN > 1;
  constexpr uint16_t mask_all = (uint16_t)((1u << CN) - 1u);
  constexpr int A_BOX_ROWS = 32, A_BOX_BYTES = A_BOX_ROWS * BK * 2;

  if (warp == 0 && lane == 0) {
    prefetch_tensormap(&tmA);
    prefetch_tensormap(&tmB);
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(bar_full + 8 * s, 1);
        mbar_init(bar_empty + 8 * s, AMC ? CN : 1);          // multicast A: every CTA of the cluster releases the stage
      }
      for (int s = 0; s < 2; ++s) {
        mbar_init(bar_tfull + 8 * s, 1);
        mbar_init(bar_tempty + 8 * s, PAIR ? 2 * EPI_WARPS : EPI_WARPS);   // PAIR: both CTAs' epilogues report to the leader
        mbar_init(bar_x + 8 * s, 1);                       // armed once per tile with the expected byte count
      }
      fence_barrier_init();
    }
    __syncwarp();
    if constexpr (PAIR) {
      tmem_alloc_2cta(tmem_slot, TMEM_COLS);
      tmem_relinquish_2cta();
    } else {
      tmem_alloc(tmem_slot, TMEM_COLS);
      tmem_relinquish();
    }
  }
  if constexpr (PAR_SMEM) {
    if (warp >= 2) {                          // the 256 epilogue threads stage one column each
      const int i = (int)threadIdx.x - 64;
      par_f[i] = p.bias[n0 + i];
      par_f[BN + i] = p.gamma[n0 + i];
      par_f[2 * BN + i] = p.beta[n0 + i];
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (CLUSTERED) cluster_sync_all();       // peers' barriers are initialised before any remote arrive
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  if (warp == 0) {
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int mb = cluster; mb < tiles_m; mb += n_clusters) {
        const int m0 = mb * ROWS + (int)rh * BM;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(bar_empty + 8 * stage, phase ^ 1);
          if constexpr (PAIR) {
            // both CTAs' bytes are counted on the leader's barrier, which only the leader arms
            const uint32_t lead_full = mapa_shared(bar_full + 8 * stage, leader);
            if (rh == 0) mbar_arrive_expect_tx(bar_full + 8 * stage, 2 * (A_STAGE_BYTES + B_BYTES));
#pragma unroll
            for (int b = 0; b < BM / A_BOX_ROWS; ++b)
              tma_load_2d_2sm(sA + stage * A_STAGE_BYTES + b * A_BOX_BYTES, &tmA, lead_full, kb * BK, m0 + b * A_BOX_ROWS);
            tma_load_2d_2sm(sB + stage * B_BYTES, &tmB, lead_full, kb * BK, n0 + (int)rh * (BN / 2));
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            continue;
          }
          mbar_arrive_expect_tx(bar_full + 8 * stage, A_STAGE_BYTES + B_STAGE_BYTES);
          tma_load_2d(sB + stage * B_STAGE_BYTES, &tmB, bar_full + 8 * stage, kb * BK, n0);
          if constexpr (AMC) {
            for (int b = (int)rank; b < BM / A_BOX_ROWS; b += CN)
              tma_load_2d_multicast(sA + stage * A_STAGE_BYTES + b * A_BOX_BYTES, &tmA, bar_full + 8 * stage, kb * BK,
                                    m0 + b * A_BOX_ROWS, mask_all);
          } else {
#pragma unroll
            for (int b = 0; b < BM / A_BOX_ROWS; ++b)
              tma_load_2d(sA + stage * A_STAGE_BYTES + b * A_BOX_BYTES, &tmA, bar_full + 8 * stage, kb * BK,
                          m0 + b * A_BOX_ROWS);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && (!PAIR || rh == 0)) {                    // PAIR: the leader issues for both CTAs
      constexpr uint32_t idesc = make_idesc_16(PAIR ? 2 * BM : BM, BN, (DT & 1) != 0, (DT & 2) != 0);
      const uint16_t mask_pair = (uint16_t)(0x3u << leader);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      for (int mb = cluster; mb < tiles_m; mb += n_clusters) {
        mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
        tcgen05_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(bar_full + 8 * stage, phase);
          tcgen05_fence_after();
          const uint32_t a_addr = sA + stage * A_STAGE_BYTES;
          const uint32_t b_addr = sB + stage * B_BYTES;
#pragma unroll
          for (int k = 0; k < BK / UMMA_K; ++k) {
            if constexpr (PAIR)
              tcgen05_mma_bf16_2cta(d_tmem, make_kmajor_sw128_desc(a_addr + k * UMMA_K * 2),
                                    make_kmajor_sw128_desc(b_addr + k * UMMA_K * 2), idesc, (kb | k) != 0 ? 1u : 0u);
            else
              tcgen05_mma_bf16(d_tmem, make_kmajor_sw128_desc(a_addr + k * UMMA_K * 2),
                               make_kmajor_sw128_desc(b_addr + k * UMMA_K * 2), idesc, (kb | k) != 0 ? 1u : 0u);
          }
          if constexpr (PAIR) tcgen05_commit_2cta_multicast(bar_empty + 8 * stage, mask_pair);
          else if constexpr (AMC) tcgen05_commit_multicast(bar_empty + 8 * stage, mask_all);
          else tcgen05_commit(bar_empty + 8 * stage);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if constexpr (PAIR) tcgen05_commit_2cta_multicast(bar_tfull + 8 * acc, mask_pair);
        else tcgen05_commit(bar_tfull + 8 * acc);
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1;
      }
    }
  } else {
    // ---------------------------------------------------------------- epilogue
    // The fp32 residual stream is stored in the "T32" blocked layout (see common.h): inside a
    // 32-row block the 16-byte column groups of the 32 rows are contiguous, so thread
    // (row = lane) reading column group g touches base + ((blk * H/4 + g) * 32 + lane) * 16:
    // every warp access is one fully coalesced 512-byte segment, straight between global memory
    // and registers in the TMEM layout (row per thread) — no staging for the residual in /
    // fp32 out traffic.
    //
    // Pass A: x = acc + bias + residual, 16 columns at a time; shifted sums give this thread's
    //         (mean, M2) over its 128 columns; x is parked back in TMEM (tcgen05.st) so that
    //         only a chunk lives in registers.
    // Exchange: every thread posts its (mean, M2) to all CTAs of the cluster (DSMEM) — 2*CN
    //         groups of 128 columns per row — and the groups are merged with Chan's formula.
    // Pass B: x back from TMEM, normalise, fp32 out (in place, coalesced), 16-bit copy through
    //         two swizzled boxes + TMA.
    const int q = warp & 3;                    // TMEM lane quarter
    const int ew = warp - 2;
    const int half = ew >> 2;                  // which 128 columns of the tile
    const int cbase = half * EPI_COLS;
    const int row_in_tile = q * 32 + lane;
    const uint32_t buf0 = sEpi + (ew * 2 + 0) * BOX_BYTES, buf1 = sEpi + (ew * 2 + 1) * BOX_BYTES;   // STAGED only
    uint32_t acc = 0, acc_phase = 0, xpar = 0, xphase0 = 0, xphase1 = 0;
    constexpr int G = 2 * CN;                  // groups of 128 columns per row
    const int groups_per_row = p.H >> 2;
    const int g0 = (n0 + cbase) >> 2;          // first 4-column group of this thread
    constexpr int NCH = EPI_COLS / 16;         // 8 chunks of 16 columns

    for (int mb = cluster; mb < tiles_m; mb += n_clusters) {
      const int m0 = mb * ROWS + (int)rh * BM;
      const int grow0 = m0 + q * 32;                         // first global row of this warp
      float4* hrow = reinterpret_cast<float4*>(p.hidden) + ((size_t)(grow0 >> 5) * groups_per_row + g0) * 32 + lane;

      // residual prefetch, four 16-column chunks deep (issued before the accumulator is ready)
      float4 rs[4][4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) rs[k][i] = hrow[(size_t)(4 * k + i) * 32];
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tcgen05_fence_after();
      const uint32_t t_addr = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + cbase;

      float pivot = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        uint32_t t[16];
        tmem_ld_x16(t_addr + 16 * j, t);
        float4 rr[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) rr[i] = rs[j & 3][i];
        if (j + 4 < NCH) {                                  // refill the slot just consumed
#pragma unroll
          for (int i = 0; i < 4; ++i) rs[j & 3][i] = hrow[(size_t)(4 * (j + 4) + i) * 32];
        }
        tcgen05_wait_ld();
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 b;
          if constexpr (PAR_SMEM) b = par4[(cbase + 16 * j) / 4 + c];
          else b = ldg_f4_ordered(p.bias + n0 + cbase + 16 * j + 4 * c);
          const float v0 = (__uint_as_float(t[4 * c + 0]) + b.x) + rr[c].x;
          const float v1 = (__uint_as_float(t[4 * c + 1]) + b.y) + rr[c].y;
          const float v2 = (__uint_as_float(t[4 * c + 2]) + b.z) + rr[c].z;
          const float v3 = (__uint_as_float(t[4 * c + 3]) + b.w) + rr[c].w;
          if (j == 0 && c == 0) pivot = v0;                  // a sample of the row: no cancellation in s2
          const float d0 = v0 - pivot, d1 = v1 - pivot, d2 = v2 - pivot, d3 = v3 - pivot;
          s1 += (d0 + d1) + (d2 + d3);
          s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
          t[4 * c + 0] = __float_as_uint(v0); t[4 * c + 1] = __float_as_uint(v1);
          t[4 * c + 2] = __float_as_uint(v2); t[4 * c + 3] = __float_as_uint(v3);
        }
        tmem_st_x16(t_addr + 16 * j, t);
      }
      tcgen05_wait_st();
      constexpr float inv_n = 1.0f / (float)EPI_COLS;
      const float mean_t = pivot + s1 * inv_n;
      const float m2_t = fmaxf(s2 - s1 * s1 * inv_n, 0.f);

      // ---- exchange (mean, M2) of the 2*CN column groups of every row
      {
        const uint32_t slot = sXchg + (uint32_t)((xpar * (2 * CN) + cg * 2 + half) * BM + row_in_tile) * 8;
        const uint32_t xb = bar_x + 8 * xpar;
        if (ew == 0 && lane == 0) mbar_arrive_expect_tx(xb, CN * EPI_WARPS * 32 * 8);   // this tile's inbox
#pragma unroll
        for (uint32_t peer = 0; peer < (uint32_t)CN; ++peer) {
          const uint32_t pr = PAIR ? 2 * peer + rh : peer;    // the CTA that holds the same rows of column group `peer`
          st_async_f32x2(mapa(slot, pr), mean_t, m2_t, mapa(xb, pr));
        }
        const uint32_t ph = xpar ? xphase1 : xphase0;
        mbar_wait(xb, ph);
        if (xpar) xphase1 ^= 1; else xphase0 ^= 1;
      }
      float mean = 0.f, M2 = 0.f;
      {
        float2 st[G];
#pragma unroll
        for (int g = 0; g < G; ++g) {
          st[g] = xchg[(xpar * (2 * CN) + g) * BM + row_in_tile];
          mean += st[g].x;
        }
        mean *= (1.0f / G);
#pragma unroll
        for (int g = 0; g < G; ++g) {
          const float d = st[g].x - mean;
          M2 += st[g].y + (float)EPI_COLS * d * d;           // Chan et al. merge of equal-size groups
        }
      }
      xpar ^= 1;
      const float rstd = rsqrtf(M2 * (1.0f / (float)(G * EPI_COLS)) + p.eps);
      const float nmr = -mean * rstd;

      // ---- pass B: fp32 back in place (T32, 512 contiguous bytes per warp access); the 16-bit
      //      operand copy is row-major for the next GEMM's TMA: each thread owns 256 contiguous
      //      bytes of its row and writes them 32 bytes per chunk.
      uint4* orow = reinterpret_cast<uint4*>(p.hidden16 + (size_t)(grow0 + lane) * p.H + n0 + cbase);
      const bool row_ok = grow0 + lane < p.M;
      if constexpr (STAGED) {
        if (lane == 0) tma_store_wait_read<0>();             // previous tile's boxes left the staging buffers
        __syncwarp();
      }
#pragma unroll
      for (int j = 0; j < NCH; ++j) {
        uint32_t t[16];
        tmem_ld_x16(t_addr + 16 * j, t);
        tcgen05_wait_ld();
        uint32_t pk[8];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float4 g4, b4;
          if constexpr (PAR_SMEM) {
            g4 = par4[(BN + cbase + 16 * j) / 4 + c];
            b4 = par4[(2 * BN + cbase + 16 * j) / 4 + c];
          } else {
            g4 = ldg_f4_ordered(p.gamma + n0 + cbase + 16 * j + 4 * c);
            b4 = ldg_f4_ordered(p.beta + n0 + cbase + 16 * j + 4 * c);
          }
          float4 y;
          y.x = fmaf(fmaf(__uint_as_float(t[4 * c + 0]), rstd, nmr), g4.x, b4.x);
          y.y = fmaf(fmaf(__uint_as_float(t[4 * c + 1]), rstd, nmr), g4.y, b4.y);
          y.z = fmaf(fmaf(__uint_as_float(t[4 * c + 2]), rstd, nmr), g4.z, b4.z);
          y.w = fmaf(fmaf(__uint_as_float(t[4 * c + 3]), rstd, nmr), g4.w, b4.w);
          hrow[(size_t)(4 * j + c) * 32] = y;
          pk[2 * c + 0] = pack16x2<FP16>(y.x, y.y);
          pk[2 * c + 1] = pack16x2<FP16>(y.z, y.w);
        }
        if constexpr (STAGED) {
          // 16 columns = 32 bytes = chunks 2*(j&3), 2*(j&3)+1 of box (j >> 2)
          const uint32_t bx = (j >> 2) ? buf1 : buf0;
          const int c16 = 2 * (j & 3);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(bx + lane * 128 + (((c16) ^ (lane & 7)) << 4)),
                       "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(bx + lane * 128 + (((c16 + 1) ^ (lane & 7)) << 4)),
                       "r"(pk[4]), "r"(pk[5]), "r"(pk[6]), "r"(pk[7]) : "memory");
        } else if (row_ok) {
          orow[2 * j + 0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
          orow[2 * j + 1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        }
      }
      // accumulator columns are free again
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (PAIR) mbar_arrive_cluster(mapa_shared(bar_tempty + 8 * acc, leader));   // the leader's MMA waits for both CTAs
        else mbar_arrive(bar_tempty + 8 * acc);
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
      if constexpr (STAGED) {
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(&tmH16, buf0, n0 + cbase, grow0);
          tma_store_2d(&tmH16, buf1, n0 + cbase + 64, grow0);
          tma_store_commit();
        }
      }
    }
    if constexpr (STAGED) {
      if (lane == 0) tma_store_wait_all();
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (CLUSTERED) cluster_sync_all();       // no CTA leaves while a peer may still address its shared memory
  if (warp == 1) {
    __syncwarp();
    tcgen05_fence_after();
    if constexpr (PAIR) tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

int tmap2d(CUtensorMap* m, const void* base, CUtensorMapDataType dt, int elt, uint64_t rows, uint64_t cols,
           uint32_t box_rows, uint32_t box_cols) {
  return get_tmap_2d(m, base, dt, elt, rows, cols, box_rows, box_cols);
}

template <int CN, int DT, bool STAGED, bool PAIR>
int launch_cn(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& t16,
              const LnParams& lp, int64_t M, cudaStream_t stream) {
  auto kern = gemm_ln_kernel<CN, DT, STAGED, PAIR>;
  constexpr int SMEM_TOTAL = smem_total<CN, STAGED, PAIR>();
  constexpr int CSIZE = PAIR ? 2 * CN : CN;
  PLLB_CUDA(opt_in_smem(kern, SMEM_TOTAL));
  cudaLaunchConfig_t cfg{};
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = SMEM_TOTAL;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CSIZE;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // persistent: as many clusters as can be co-resident (clusters must fit inside a GPC)
  static thread_local int max_clusters[MAX_CN + 1][32] = {};
  int& mc = max_clusters[CN][DT + (STAGED ? 8 : 0) + (PAIR ? 16 : 0)];
  if (mc == 0) {
    cfg.gridDim = dim3(CSIZE * (sm_count() / CSIZE));
    int n = 0;
    cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
    if (e != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = sm_count() / CSIZE;
    }
    mc = n;
  }
  const int64_t tiles_m = ceil_div(M, PAIR ? 2 * BM : BM);
  const int clusters = (int)(tiles_m < mc ? tiles_m : mc);
  cfg.gridDim = dim3(CSIZE * clusters);
  PLLB_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, t16, lp));
  ++g_launch_counter;
  return PLLB_OK;
}

template <int CN, int DT>
int launch_cn_dt(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& t16, const LnParams& lp, int64_t M,
                 bool staged, bool pair, cudaStream_t stream) {
  if (pair) return staged ? launch_cn<CN, DT, true, true>(ta, tb, t16, lp, M, stream)
                          : launch_cn<CN, DT, false, true>(ta, tb, t16, lp, M, stream);
  return staged ? launch_cn<CN, DT, true, false>(ta, tb, t16, lp, M, stream)
                : launch_cn<CN, DT, false, false>(ta, tb, t16, lp, M, stream);
}

}  // namespace

int launch_gemm_ln(const void* A, const void* W, const float* bias, const float* gamma, const float* beta, float eps,
                   float* hidden_f32, void* hidden_16, int64_t M, int H, int K, int dt, cudaStream_t stream) {
  if (M <= 0) return PLLB_OK;
  if (H % BN != 0 || H / BN > MAX_CN || K % BK != 0 || M > INT32_MAX)
    return fail(PLLB_ERR_INVALID, "gemm_ln: need H in {256,512,768,1024} and K % 64 == 0");
  // epilogue-paced (K <= H): staged 16-bit output; mainloop-paced (K > H): deeper operand ring
  const bool staged = K <= H;
  // cta_group::2 pairs inside the LayerNorm cluster (PLLB_LN_PAIR: 0 never, 1 default policy, 2 always).
  // Default: the mainloop-paced launches (K > H, i.e. FFN2) for H = 256 (cluster 2: 148 SMs), H = 768
  // (cluster 6: 132 SMs against 135; measured FFN2 -15.5 %, C2 step -3.0 %) and H = 1024 (cluster 8: 120
  // SMs against 132; measured FFN2 -8.7 %, C4 step -2.0 %).  H = 512 would drop from 148 to 132 SMs
  // and is left unpaired (no model of that width was measured).
  const char* pe = getenv("PLLB_LN_PAIR");
  const int pair_policy = pe ? atoi(pe) : 1;
  const int cn = H / BN;
  const bool mainloop_paced = K > H;
  const bool pair = M > 2 * BM && (pair_policy == 2 || (pair_policy == 1 && mainloop_paced && cn != 2));
  CUtensorMap ta, tb, t16;
  int rc;
  if ((rc = tmap2d(&ta, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)M, (uint64_t)K, 32, BK))) return rc;   // 32-row boxes
  if ((rc = tmap2d(&tb, W, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)H, (uint64_t)K, pair ? BN / 2 : BN, BK))) return rc;
  if ((rc = tmap2d(&t16, hidden_16, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (uint64_t)M, (uint64_t)H, 32, 64))) return rc;
  LnParams lp{(int)M, K, H, hidden_f32, reinterpret_cast<__nv_bfloat16*>(hidden_16), bias, gamma, beta, eps};
#define PLLB_LN(CN_)                                                                                          \
  case CN_:                                                                                                   \
    switch (dt) {                                                                                             \
      case DT_BF16: return launch_cn_dt<CN_, DT_BF16>(ta, tb, t16, lp, M, staged, pair, stream);              \
      case DT_BF16_OUT16: return launch_cn_dt<CN_, DT_BF16_OUT16>(ta, tb, t16, lp, M, staged, pair, stream);  \
      case DT_FP16: return launch_cn_dt<CN_, DT_FP16>(ta, tb, t16, lp, M, staged, pair, stream);              \
    }                                                                                                         \
    return fail(PLLB_ERR_INVALID, "gemm_ln: unsupported operand dtype combination");
  switch (cn) {
    PLLB_LN(1)
    PLLB_LN(2)
    PLLB_LN(3)
    PLLB_LN(4)
  }
#undef PLLB_LN
  return fail(PLLB_ERR_INVALID, "gemm_ln: unsupported hidden size");
}

}  // namespace pllb
