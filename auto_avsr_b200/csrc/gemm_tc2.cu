// Two-SM tensor-core GEMM (tcgen05 cta_group::2) for the FFN projections: y = [resid + alpha *] act(x W^T + b).
//
// Why: the r01 profiles show the 1-CTA kernel's main loop is bound by what one SM can ingest through TMA
// (~46 B/cycle), not by the tensor pipe.  A CTA PAIR (thread-block cluster of 2 on one TPC) computes a 256 x BNP
// tile with ONE tcgen05.mma.cta_group::2 stream issued by the leader CTA: each CTA stages only its own 128 rows of
// A and HALF of the B rows (the MMA reads the other half from the peer's shared memory), so per SM the bytes per
// MAC halve compared with a 128 x 128 tile and the tensor pipe stays ~balanced with the ingest port
// (FFN w_1, pair tile 256 x 512: 48 KB per k-block per SM = 1043 cycles of ingest vs 1024 cycles of MMA).
//
// Structure per CTA (320 threads): warp 0 TMA producer (both CTAs; 2-SM TMA signals the LEADER's `full` barrier),
// warp 1 MMA issuer (leader only) + TMEM allocation (both, cta_group::2), warps 2-9 epilogue (both; each CTA drains
// the 128 accumulator rows that live in its own TMEM through the same staged, coalesced epilogue as gemm_tc.cu).
// One pair-tile per cluster (the FFN shapes give 42 pair-tiles <= 74 pairs), so no accumulator double buffering.
// fp16 operands, EPI_LINEAR only; everything else uses gemm_tc.cu.
#include "common.cuh"
#include "epilogue.cuh"
#include "sm100.cuh"

namespace avsr {

using namespace sm100;

constexpr int T2_THREADS = 320;
constexpr int T2_STG_WARP = STG_WARP;
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;   // shared::cluster address with the CTA-pair peer bit cleared = leader CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster.  Relaxed: what the arrival
// publishes is tensor-memory state, ordered by tcgen05.wait::st + tcgen05.fence::before_thread_sync on this side and
// tcgen05.fence::after_thread_sync on the waiter's; a release at cluster scope costs a MEMBAR.ALL.GPU per arrival
// (r02 trace: the first MMA of the 384-wide tile started 1400 cycles late behind 16 of them).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(bar), "r"(rank));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {   // acquire at cluster scope
  uint32_t spins = 0, ok = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) break;
    if (++spins > (1u << 24)) __trap();
  }
}
template <int COLS>
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t dst_smem) {  // one warp in EACH CTA of the pair, same dst offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "n"(COLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS) : "memory");
}
// 2-SM TMA load: data lands in THIS CTA's shared memory, completion bytes are credited to the LEADER CTA's barrier
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* m, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      :
      : "r"(dst), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// D[tmem, both CTAs] (+)= A[256 rows: 128 per CTA] * B[N: N/2 rows per CTA]^T, issued by the leader CTA only
__device__ __forceinline__ void mma_f16_2sm(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all MMAs issued so far -> arrive on the barrier at the same offset in BOTH CTAs of the pair
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}

// A pair tile of width BNP is covered by up to two MMA sub-blocks (UMMA N <= 256): 128 -> {128}, 256 -> {256},
// 384 -> {256, 128}, 512 -> {256, 256}.  Each CTA stages half of every sub-block's B rows.
template <int BNP, int MODE = EPI_LINEAR, bool RESID = false>
struct T2Cfg {
  static constexpr int kNSub = BNP > 256 ? 2 : 1;
  static constexpr int kN0 = BNP > 256 ? 256 : BNP;              // width of sub-block 0
  static constexpr int kN1 = BNP > 256 ? BNP - 256 : 0;          // width of sub-block 1 (0, 128 or 256)
  static constexpr int kBRowsTotal = BNP / 2;                    // B rows per CTA per stage
  static constexpr int kABytes = 128 * 128;
  static constexpr int kBBytes = kBRowsTotal * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;          // per CTA
  static constexpr int kVecBytes = 3 * BNP * 4;   // bias / pos_bias_u / pos_bias_v of the tile's columns
  // EPI_LINEAR leaves through TMA stores staged in the pipeline stages (idle once the accumulator is complete) or, with
  // a residual, in the TMA-prefetched residual tile itself; the other modes keep the transposing staging buffers
  static constexpr int kStgBytes = MODE == EPI_LINEAR ? 0 : 8 * T2_STG_WARP;
  static constexpr int kResBytes = RESID ? 128 * BNP * 4 : 0;    // this CTA's 128 x BNP fp32 residual tile
  static constexpr int kFixed = 1024 + 256 + kVecBytes + kStgBytes + kResBytes;
  static constexpr int kStagesFit = (222 * 1024 - kFixed) / kStageBytes;
  static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
  static constexpr int kSmem = kStages * kStageBytes + kFixed;
  static constexpr int kTmemCols = BNP <= 128 ? 128 : (BNP <= 256 ? 256 : 512);
  static_assert(kStages >= 2 && BNP % 32 == 0 && BNP <= 512, "bad pair tile");
  static_assert(MODE != EPI_LINEAR || kStages * kStageBytes >= 8 * 16384, "LINEAR staging (8 warps x 4 x 4 KB) lives in the stages");
  __host__ __device__ static constexpr int sub_n(int j) { return j == 0 ? kN0 : kN1; }
  __host__ __device__ static constexpr int sub_col(int j) { return j == 0 ? 0 : kN0; }          // first tile column
  __host__ __device__ static constexpr int sub_brow(int j) { return j == 0 ? 0 : kN0 / 2; }     // first B smem row
};

// -DAVSR_TRACE_EPI (with -DAVSR_TRACE): marks 2..5 and 9 are taken by the first epilogue warp instead of the producer / MMA
// warps: 2 first chunk in registers, 3 first chunk staged, 4 first store issued, 5 last store issued, 9 reserved
#if defined(AVSR_TRACE) && defined(AVSR_TRACE_EPI)
#define T2_PMARK(cond, s) do { } while (0)
#define T2_EMARK(s) AVSR_TRACE_MARK(threadIdx.x == 64, trc, s)
#else
#define T2_PMARK(cond, s) AVSR_TRACE_MARK(cond, trc, s)
#define T2_EMARK(s) do { } while (0)
#endif

// RELU / RESID are compile-time: a predicated-off instruction still takes an issue slot, and this epilogue is not
// overlapped with anything (one tile per cluster).
// PREB (inside the encoder forward, whose B operands are prepared weights; +0.6 % in the r02 A/B): the B operand does
// not depend on the predecessor kernel, so the producer fills the B halves of the first stages BEFORE
// griddepcontrol.wait; after the wait only the A tiles (just written by the predecessor, L2-resident) are still to come.
template <int MODE, int BNP, bool RELU, bool RESID, bool PREB = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(T2_THREADS, 1)
gemm_tc2_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmB1, const __grid_constant__ CUtensorMap tmOut,
                const __grid_constant__ CUtensorMap tmRes, int K, int tiles_n, int nsplit, EpiParams ep) {
  using Cfg = T2Cfg<BNP, MODE, RESID>;
  constexpr int S = Cfg::kStages;
  constexpr int KE = 64;   // halves per 128-byte k-block
  extern __shared__ uint8_t t2_smem_raw[];
  const uint32_t raw = smem_u32(t2_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* gen = t2_smem_raw + (base - raw);
  // [stages][residual tile (RESID)][barriers 256 B][per-column vectors][staging (non-LINEAR modes)]
  constexpr int kBarOff = S * Cfg::kStageBytes + Cfg::kResBytes;
  const uint32_t res_base = base + S * Cfg::kStageBytes;
  const uint32_t bars = base + kBarOff;   // full[S], empty[S], tmem_full, (tmem slot), res_full
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + kBarOff + (2 * S + 1) * 8);
  const uint32_t res_full_bar = bars + 8u * (2 * S + 2);
  const uint32_t acc_ready_bar = bars + 8u * (2 * S + 3);   // leader's: the 16 epilogue warps of the pair pre-filled the accumulator
  float* s_bias = reinterpret_cast<float*>(gen + kBarOff + 256);
  uint8_t* stg_base = gen + kBarOff + 256 + Cfg::kVecBytes;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (S + s); };
  const uint32_t tmem_full_bar = bars + 8u * (2 * S);
#ifdef AVSR_TRACE
  // phase marks: 0 prologue done, 1 dependency resolved, 2 first TMA issued, 3 last TMA issued, 4 first stage full,
  // 5 last MMA committed, 6 accumulator visible to the epilogue, 7 epilogue warp done, 8 cluster drained
  unsigned long long** trc = reinterpret_cast<unsigned long long**>(gen + kBarOff + 192);
  if (threadIdx.x == 0) AVSR_TRACE_OPEN(trc, 200 + MODE, (unsigned)BNP | ((unsigned)(K / 64 / nsplit) << 16));
#endif

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();          // 0 = leader
  // nsplit > 1 (deferred split-K): cluster = (pair-tile, k-slice); the slice's raw fp32 accumulators go to
  // out + slice * M * ldo and the consumer (the following LayerNorm) sums the slices in a fixed order
  const int cl = blockIdx.x >> 1;
  const int pair = cl / nsplit, split = cl - pair * nsplit;
  const int m0 = (pair / tiles_n) * 256, n0 = (pair % tiles_n) * BNP;
  const int nkb = K / KE / nsplit;
  const int kb0 = split * nkb;

  pdl_launch_dependents();
  // PREB: the per-column vectors are fetched into registers now, so that their latency is spent under the prologue's
  // barrier set-up / TMEM allocation / cluster sync instead of in front of the accumulator pre-fill
  const bool has_bias = ep.bias != nullptr;
  constexpr int kVecPer = (BNP + (T2_THREADS - 64) - 1) / (T2_THREADS - 64);
  float vpre[MODE == EPI_QK ? 3 : 1][kVecPer];
  auto fetch_vectors = [&]() {
#pragma unroll
    for (int i = 0; i < kVecPer; ++i) {
      const int c = (int)threadIdx.x - 64 + i * (T2_THREADS - 64);
      const int n = n0 + c;
      vpre[0][i] = (has_bias && c < BNP && n < ep.N) ? ep.bias[n] : 0.f;
      if constexpr (MODE == EPI_QK) {
        const bool isq = c < BNP && n < ep.H * kHeadDim;
        vpre[1][i] = isq ? ep.pos_u[n] : 0.f;
        vpre[2][i] = isq ? ep.pos_v[n] : 0.f;
      }
    }
  };
  if constexpr (PREB) {
    if (warp >= 2) fetch_vectors();
  }
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if constexpr (Cfg::kNSub == 2) tma_prefetch_desc(&tmB1);
    for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    mbar_init(tmem_full_bar, 1);
    mbar_init(res_full_bar, 1);
    mbar_init(acc_ready_bar, 16);
    if constexpr (MODE == EPI_LINEAR) { tma_prefetch_desc(&tmOut); if (RESID) tma_prefetch_desc(&tmRes); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2sm<Cfg::kTmemCols>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // both CTAs' barriers are initialised and TMEM is allocated before anyone signals a peer
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  AVSR_TRACE_MARK(threadIdx.x == 0, trc, 0);
  // Producer and MMA warps run warp-uniform loops and guard only the instruction issue with elect.sync: TMA / tcgen05
  // operands live in uniform registers, and inside a divergent `lane == 0` region every operand is rebuilt and moved
  // per instruction (r02 SASS: ~22 instructions + an ELECT / BRA.U.ANY loop per UTCHMMA).
  // The bias is not added in the epilogue: the epilogue warps, idle until the accumulator is complete, write it into the
  // accumulator (TMEM column c of every row = bias[n0 + c]) while the pipeline fills, and the MMAs accumulate on top --
  // r02 epilogue trace: 206 instructions per 64-column chunk, 64 of them the bias FADDs behind 16 dependent LDS.128.
  auto stage_vectors_and_prefill = [&]() {
    if constexpr (!PREB) fetch_vectors();
#pragma unroll
    for (int i = 0; i < kVecPer; ++i) {
      const int c = (int)threadIdx.x - 64 + i * (T2_THREADS - 64);
      if (c < BNP) {
        s_bias[c] = vpre[0][i];
        if constexpr (MODE == EPI_QK) {
          s_bias[BNP + c] = vpre[1][i];
          s_bias[2 * BNP + c] = vpre[2][i];
        }
      }
    }
    asm volatile("bar.sync 1, 256;" ::: "memory");
    if (has_bias) {
      const int q = warp & 3, chalf = (warp - 2) >> 2;
      const int cb = (BNP == 96) ? chalf * 64 : chalf * (BNP / 2);
      const int ce = (BNP == 96) ? (chalf ? 96 : 64) : cb + BNP / 2;
      const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll 1
      for (int c = cb; c < ce; c += 32) {
        float bv[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 t = *reinterpret_cast<const float4*>(s_bias + c + 4 * j);
          bv[4 * j] = t.x; bv[4 * j + 1] = t.y; bv[4 * j + 2] = t.z; bv[4 * j + 3] = t.w;
        }
        tmem_st32(trow + c, bv);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (elect_one_sync()) mbar_arrive_cluster(acc_ready_bar, 0);
    }
  };
  if constexpr (PREB) {          // prepared weights: the bias does not depend on the predecessor either
    if (warp >= 2) stage_vectors_and_prefill();
  }
  if constexpr (PREB) {
    if (warp == 0) {
      const int npre = nkb < S ? nkb : S;      // every stage is free on entry: no empty-barrier wait needed
      for (int kb = 0; kb < npre; ++kb) {
        if (elect_one_sync()) {
          if (rank == 0) mbar_expect_tx(full_bar(kb), 2 * Cfg::kStageBytes);
          const uint32_t dst = base + kb * Cfg::kStageBytes;
          const int kc = (kb0 + kb) * KE;
          tma_load_2d_2sm(dst + Cfg::kABytes, &tmB, kc, n0 + (int)rank * (Cfg::kN0 / 2), full_bar(kb));
          if constexpr (Cfg::kNSub == 2)
            tma_load_2d_2sm(dst + Cfg::kABytes + Cfg::sub_brow(1) * 128, &tmB1, kc,
                            n0 + Cfg::kN0 + (int)rank * (Cfg::kN1 / 2), full_bar(kb));
        }
      }
    }
  }
  pdl_wait();
  AVSR_TRACE_MARK(threadIdx.x == 0, trc, 1);
  AVSR_TRACE_STAMP(threadIdx.x == 0, trc, 10);
  if constexpr (!PREB) {
    if (warp >= 2) stage_vectors_and_prefill();
  }

  if (warp == 0) {
    if constexpr (RESID) {
      // this CTA's 128 x BNP tile of the residual stream (complete before the predecessor started): fetched now, consumed
      // -- and overwritten in place -- by the epilogue, which stores the updated tile from the same shared memory
      if (elect_one_sync()) {
        mbar_expect_tx(res_full_bar, Cfg::kResBytes);
#pragma unroll
        for (int j = 0; j < BNP / 32; ++j)
          tma_load_2d(res_base + j * (128 * 128), &tmRes, n0 + 32 * j, m0 + (int)rank * 128, res_full_bar);
      }
    }
    for (int kb = 0; kb < nkb; ++kb) {
      const int s = kb % S;
      const uint32_t ph = (kb / S) & 1;
      if constexpr (PREB) {
        if (kb < S) {                                                   // expect_tx + B already issued before the wait
          if (elect_one_sync())
            tma_load_2d_2sm(base + s * Cfg::kStageBytes, &tmA, (kb0 + kb) * KE, m0 + (int)rank * 128, full_bar(s));
          T2_PMARK(kb == 0 && lane == 0, 2);
          continue;
        }
      }
      mbar_wait(empty_bar(s), ph ^ 1);                                  // own stage free (leader's commit, multicast)
      if (elect_one_sync()) {
        if (rank == 0) mbar_expect_tx(full_bar(s), 2 * Cfg::kStageBytes); // bytes of BOTH CTAs land on the leader's barrier
        const uint32_t dst = base + s * Cfg::kStageBytes;
        const int kc = (kb0 + kb) * KE;
        tma_load_2d_2sm(dst, &tmA, kc, m0 + (int)rank * 128, full_bar(s));
        // sub-block 0 with box tmB (kN0/2 rows), sub-block 1 with box tmB1 (kN1/2 rows)
        tma_load_2d_2sm(dst + Cfg::kABytes, &tmB, kc, n0 + (int)rank * (Cfg::kN0 / 2), full_bar(s));
        if constexpr (Cfg::kNSub == 2)
          tma_load_2d_2sm(dst + Cfg::kABytes + Cfg::sub_brow(1) * 128, &tmB1, kc,
                          n0 + Cfg::kN0 + (int)rank * (Cfg::kN1 / 2), full_bar(s));
      }
      T2_PMARK(kb == 0 && lane == 0, 2);
    }
    T2_PMARK(lane == 0, 3);
  } else if (warp == 1) {
    if (rank == 0) {
      constexpr uint32_t idesc0 = umma_idesc_f16(256, Cfg::kN0);
      constexpr uint32_t idesc1 = umma_idesc_f16(256, Cfg::kNSub == 2 ? Cfg::kN1 : Cfg::kN0);
      const uint32_t acc0 = has_bias ? 1u : 0u;          // pre-filled accumulator: the first MMA accumulates too
      if (has_bias) {
        mbar_wait_cluster(acc_ready_bar, 0);
        tc_fence_after();
      }
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb % S;
        const uint32_t ph = (kb / S) & 1;
        mbar_wait(full_bar(s), ph);
        tc_fence_after();
        T2_PMARK(kb == 0 && lane == 0, 4);
        const uint32_t a_addr = base + s * Cfg::kStageBytes;
        const uint64_t a_desc = umma_desc_sw128(a_addr);
        if (elect_one_sync()) {
#pragma unroll
          for (int j = 0; j < Cfg::kNSub; ++j) {
            const uint64_t b_desc = umma_desc_sw128(a_addr + Cfg::kABytes + Cfg::sub_brow(j) * 128);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              mma_f16_2sm(tmem_base + Cfg::sub_col(j), a_desc + 2 * k, b_desc + 2 * k, j == 0 ? idesc0 : idesc1, acc0 | (uint32_t)((kb | k) != 0));
          }
          tc_commit_2sm(empty_bar(s));       // frees the stage in both CTAs
          if (kb == nkb - 1) tc_commit_2sm(tmem_full_bar);   // accumulator complete: wakes both CTAs' epilogues
        }
      }
      T2_PMARK(lane == 0, 5);
    }
  } else {
    // ---------------------------------------------------------------- epilogue (both CTAs: own 128 rows)
    const int q = warp & 3;
    const int chalf = (warp - 2) >> 2;
    uint8_t* stg = stg_base + (warp - 2) * T2_STG_WARP;
    // column ranges of the two warps that share a lane quarter (whole 32-column chunks; 96 = 64 + 32)
    const int cb = (BNP == 96) ? chalf * 64 : chalf * (BNP / 2);
    const int ce = (BNP == 96) ? (chalf ? 96 : 64) : cb + BNP / 2;
    const int pr = lane >> 3, pc = lane & 7;
    mbar_wait(tmem_full_bar, 0);
    tc_fence_after();
    AVSR_TRACE_MARK(threadIdx.x == 64, trc, 6);
    const int mw = m0 + (int)rank * 128 + q * 32;
    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16);
    if constexpr (MODE == EPI_GLU) {
      // interleaved pointwise_cov1: per 128-column group, value columns [g, g+64), their gates 64 further
#pragma unroll 1
      for (int g = 0; g < BNP; g += 128) {
        const int c = g + chalf * 32;
        float val[32], gate[32];
        tmem_ld32(trow + c, val);
        tmem_ld32(trow + c + 64, gate);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) val[j] *= sigmoidf_fast(gate[j]);
        stage_write_f32(stg, lane, val, false);
        __syncwarp();
#pragma unroll
        for (int it = 0; it < 8; ++it) emit_glu(ep, mw + it * 4 + pr, n0 + c + pc * 4, stage_read(stg, it, lane));
        __syncwarp();
      }
    } else if constexpr (MODE == EPI_QK) {
      const int D = ep.H * kHeadDim;
#pragma unroll 1
      for (int c = cb; c < ce; c += 64) {
        float v[64];
        tmem_ld32(trow + c, v);
        tmem_ld32(trow + c + 32, v + 32);
        tmem_ld_wait();
        const int n = n0 + c;
        const int np = n + pc * 8;
        const int seg = np / D, nn = np - seg * D;
        const int hh = nn >> 6, d0 = nn & 63;
        int rb[8], rt[8];
        bool rok[8];
        {
          const int mrow = mw + pr;
          int bb = mrow / ep.T, tt = mrow - bb * ep.T;
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            rb[it] = bb; rt[it] = tt; rok[it] = (mrow + it * 4 < ep.M) && (np < ep.N);
            tt += 4;
            while (tt >= ep.T) { tt -= ep.T; ++bb; }
          }
        }
        if (n < D) {                                       // q: q + pos_bias_u and q + pos_bias_v
          const float* su = s_bias + BNP + c;
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] += su[j];
          stage_write_f16(stg, lane, v);
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 8; ++it)
            emit_heads<__half>(ep, ep.qu, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
          __syncwarp();
          tmem_ld32(trow + c, v);
          tmem_ld32(trow + c + 32, v + 32);
          tmem_ld_wait();
          const float* sv = s_bias + 2 * BNP + c;
#pragma unroll
          for (int j = 0; j < 64; ++j) v[j] += sv[j];
          stage_write_f16(stg, lane, v);
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 8; ++it)
            emit_heads<__half>(ep, ep.qv, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
          __syncwarp();
        } else {
          stage_write_f16(stg, lane, v);
          __syncwarp();
          void* dst = n < 2 * D ? ep.kk : ep.vt;
#pragma unroll
          for (int it = 0; it < 8; ++it)
            emit_heads<__half>(ep, dst, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
          __syncwarp();
        }
      }
    } else if constexpr (MODE == EPI_LSE) {                // fp32 logits + log-sum-exp partials of the valid columns
      float* outp = reinterpret_cast<float*>(ep.out);
      float rm = -INFINITY, rs = 0.f;                      // this thread's row: running max, sum of exp(x - max)
      int ri = 0x7fffffff;                                 // first index of the running max
#pragma unroll 1
      for (int c = cb; c < ce; c += 32) {
        float v[32];
        tmem_ld32(trow + c, v);
        tmem_ld_wait();
        const int nb = n0 + c;
        if (nb < ep.n_valid) {
          const int nv = ep.n_valid - nb;                  // valid columns of this chunk (>= 32: all)
          float cm = -INFINITY;
          int ci = 0;
#pragma unroll
          for (int j = 0; j < 32; ++j)
            if (j < nv && v[j] > cm) { cm = v[j]; ci = j; }
          if (cm > rm) { rs *= __expf(rm - cm); rm = cm; ri = nb + ci; }   // rm = -inf: rs is 0, exp(-inf) = 0
          float acc = 0.f;
#pragma unroll
          for (int j = 0; j < 32; ++j) acc += (j < nv) ? __expf(v[j] - rm) : 0.f;
          rs += acc;
        }
        stage_write_f32(stg, lane, v, false);
        __syncwarp();
        const int n = n0 + c + pc * 4;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int m = mw + it * 4 + pr;
          const uint4 pay = stage_read(stg, it, lane);
          if (m < ep.M && n < ep.N) *reinterpret_cast<uint4*>(outp + (long)m * ep.ldo + n) = pay;
        }
        __syncwarp();
      }
      const int row = mw + lane;
      if (row < ep.M) {
        LsePart pt;
        pt.m = rm; pt.s = rs; pt.idx = ri; pt.pad = 0;
        ep.lse_part[(long)((n0 / BNP) * 2 + chalf) * ep.M + row] = pt;
      }
    } else if (!ep.round_out) {                            // fp32 destination (+ residual)
      // lane = accumulator row.  Each 32-column chunk is a [32 rows][128 B] box in the TMA 128-byte swizzle (16-byte piece
      // j of row r at piece j ^ (r & 7): conflict-free lane-per-row accesses, no padding) that ONE TMA store writes out
      // (rows >= M clipped by the tensor map) -- no transposing read-back, no per-lane addressing or bounds tests.
      const int mrow = m0 + (int)rank * 128 + q * 32;
      const uint32_t sw = (uint32_t)(lane & 7);
      if constexpr (RESID) {
        // the chunk's box is the matching piece of the prefetched residual tile: x += alpha * (acc + b) in place
        mbar_wait(res_full_bar, 0);
#pragma unroll 1
        for (int c = cb; c < ce; c += 32) {
          float v[32];
          tmem_ld32(trow + c, v);
          uint8_t* box = gen + S * Cfg::kStageBytes + (c >> 5) * (128 * 128) + q * 4096;
          float4 r[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) r[j] = *reinterpret_cast<const float4*>(box + lane * 128 + ((j ^ sw) << 4));
          tmem_ld_wait();
          if (c == cb) T2_EMARK(2);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            r[j].x = fmaf(ep.alpha, v[4 * j], r[j].x); r[j].y = fmaf(ep.alpha, v[4 * j + 1], r[j].y);
            r[j].z = fmaf(ep.alpha, v[4 * j + 2], r[j].z); r[j].w = fmaf(ep.alpha, v[4 * j + 3], r[j].w);
            *reinterpret_cast<float4*>(box + lane * 128 + ((j ^ sw) << 4)) = r[j];
          }
          fence_proxy_async();
          __syncwarp();
          if (c == cb) T2_EMARK(3);
          if (elect_one_sync()) {
            tma_store_3d(&tmOut, res_base + (c >> 5) * (128 * 128) + q * 4096, n0 + c, mrow, split);
            tma_store_commit();
          }
          if (c == cb) T2_EMARK(4);
          if (c + 32 >= ce) T2_EMARK(5);
        }
      } else {
        // staging: a ring of four 4 KB boxes per warp in the (now idle) pipeline stages -- the export, not the
        // conversion, bounds this epilogue (r02 trace), so the stores are queued as early as the data exists
        const uint32_t stg0 = base + (uint32_t)(warp - 2) * 16384u;
#pragma unroll 1
        for (int c = cb, ci = 0; c < ce; c += 32, ++ci) {
          float v[32];
          tmem_ld32(trow + c, v);
          if (ci >= 4) {                                   // the box is free once its previous store has been read
            if (elect_one_sync()) tma_store_wait_read_n<3>();
            __syncwarp();
          }
          tmem_ld_wait();
          uint8_t* box = gen + (warp - 2) * 16384 + (ci & 3) * 4096;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            if (RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            *reinterpret_cast<float4*>(box + lane * 128 + ((j ^ sw) << 4)) = o;
          }
          fence_proxy_async();
          __syncwarp();
          if (elect_one_sync()) {
            tma_store_3d(&tmOut, stg0 + (uint32_t)(ci & 3) * 4096u, n0 + c, mrow, split);
            tma_store_commit();
          }
        }
      }
      if (elect_one_sync()) tma_store_wait_read_n<0>();    // shared memory must outlive the stores' reads
    } else {                                               // fp16 operand destination (FFN hidden)
      // 64-column chunks = [32 rows][128 B] boxes of halves, same staging / TMA-store scheme; the tcgen05.ld of chunk
      // i+1 is in flight while chunk i is converted and staged
      constexpr int NC = (BNP / 2) / 64;                   // 64-column chunks per warp (4 for the 256x512 pair tile)
      const int mrow = m0 + (int)rank * 128 + q * 32;
      const uint32_t sw = (uint32_t)(lane & 7);
      const uint32_t stg0 = base + (uint32_t)(warp - 2) * 16384u;
      static_assert(NC <= 4, "one staging box per chunk");
      float va[64], vb[64];
      tmem_ld32(trow + cb, va);
      tmem_ld32(trow + cb + 32, va + 32);
#pragma unroll
      for (int ci = 0; ci < NC; ++ci) {
        const int c = cb + ci * 64;
        float* v = (ci & 1) ? vb : va;
        float* vn = (ci & 1) ? va : vb;
        tmem_ld_wait();
        if (ci == 0) T2_EMARK(2);
        if (ci + 1 < NC) {
          tmem_ld32(trow + c + 64, vn);
          tmem_ld32(trow + c + 96, vn + 32);
        }
        uint8_t* box = gen + (warp - 2) * 16384 + ci * 4096;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          uint32_t pk[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float a = v[8 * j + 2 * e], b = v[8 * j + 2 * e + 1];
            pk[e] = RELU ? pack_half2_sat_relu(a, b) : pack_half2_sat(a, b);
          }
          *reinterpret_cast<uint4*>(box + lane * 128 + ((j ^ sw) << 4)) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        }
        fence_proxy_async();
        __syncwarp();
        if (ci == 0) T2_EMARK(3);
        if (elect_one_sync()) {
          tma_store_3d(&tmOut, stg0 + (uint32_t)ci * 4096u, n0 + c, mrow, split);
          tma_store_commit();
        }
        if (ci == 0) T2_EMARK(4);
        if (ci == NC - 1) T2_EMARK(5);
      }
      if (elect_one_sync()) tma_store_wait_read_n<0>();
    }
  }
  AVSR_TRACE_MARK(threadIdx.x == 64, trc, 7);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();          // the peer may still be reading TMEM / its barriers may still receive our commits
  AVSR_TRACE_MARK(threadIdx.x == 0, trc, 8);
  AVSR_TRACE_STAMP(threadIdx.x == 0, trc, 11);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_2sm<Cfg::kTmemCols>(tmem_base);
  }
}

AVSR_TRACE_DEFINE_BIND(trace_bind_gemm_tc2)

// set by encoder.cu around the forward schedule: B operands are prepared weights nobody writes during the forward
thread_local bool g_tc2_weights_static = false;

template <int MODE, int BNP, bool RELU, bool RESID>
static int launch_tc2_k(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmB1, const CUtensorMap& tmOut,
                        const CUtensorMap& tmRes, int grid, int K, int tiles_n, int nsplit, const EpiParams& ep,
                        cudaStream_t st) {
  using Cfg = T2Cfg<BNP, MODE, RESID>;
  AVSR_SET_MAX_SMEM((gemm_tc2_kernel<MODE, BNP, RELU, RESID>), Cfg::kSmem);
  const EpiParams& epl = ep;
  if (g_tc2_weights_static) {
    AVSR_SET_MAX_SMEM((gemm_tc2_kernel<MODE, BNP, RELU, RESID, true>), Cfg::kSmem);
    AVSR_LAUNCH((gemm_tc2_kernel<MODE, BNP, RELU, RESID, true>), grid, T2_THREADS, Cfg::kSmem, st, tmA, tmB, tmB1, tmOut,
                tmRes, K, tiles_n, nsplit, epl);
    return AVSR_OK;
  }
  AVSR_LAUNCH((gemm_tc2_kernel<MODE, BNP, RELU, RESID>), grid, T2_THREADS, Cfg::kSmem, st, tmA, tmB, tmB1, tmOut, tmRes, K,
              tiles_n, nsplit, epl);
  return AVSR_OK;
}

template <int MODE, int BNP>
static int launch_tc2(const __half* A, const __half* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st,
                      int nsplit = 1) {
  using Cfg = T2Cfg<BNP>;
  CUtensorMap tmA, tmB, tmB1;
  AVSR_TRY(make_tmap_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, 128, 2));
  AVSR_TRY(make_tmap_2d(&tmB, Bw, (uint64_t)N, (uint64_t)K, (uint64_t)K, Cfg::kN0 / 2, 2));
  AVSR_TRY(make_tmap_2d(&tmB1, Bw, (uint64_t)N, (uint64_t)K, (uint64_t)K, Cfg::kNSub == 2 ? Cfg::kN1 / 2 : Cfg::kN0 / 2, 2));
  const int tiles_m = cdiv(M, 256), tiles_n = cdiv(N, BNP);
  const int grid = 2 * tiles_m * tiles_n * nsplit;
  CUtensorMap tmOut = tmA, tmRes = tmA;    // only EPI_LINEAR reads them
  if constexpr (MODE == EPI_LINEAR) {
    // output as a (k-slice, row, column) tensor with [1][32 rows][128 B] store boxes: rows >= M are clipped per slice
    const int esz = ep.round_out ? 2 : 4;
    AVSR_TRY(make_tmap_3d(&tmOut, ep.out, (uint64_t)nsplit, (uint64_t)M, (uint64_t)N, (uint64_t)ep.ldo,
                          (uint64_t)M * (uint64_t)ep.ldo, 32, esz));
    const bool relu = ep.relu != 0, resid = ep.resid != nullptr;
    if (resid) {
      AVSR_REQUIRE(!ep.round_out && nsplit == 1 && BNP == 128, "two-SM GEMM: the residual epilogue is fp32, unsplit, 256x128 tiles");
      AVSR_TRY(make_tmap_2d(&tmRes, ep.resid, (uint64_t)M, (uint64_t)N, (uint64_t)ep.ldo, 128, 4));
    }
    if constexpr (BNP == 128) {
      if (relu && resid) return launch_tc2_k<MODE, BNP, true, true>(tmA, tmB, tmB1, tmOut, tmRes, grid, K, tiles_n, nsplit, ep, st);
      if (resid) return launch_tc2_k<MODE, BNP, false, true>(tmA, tmB, tmB1, tmOut, tmRes, grid, K, tiles_n, nsplit, ep, st);
    }
    if (relu) return launch_tc2_k<MODE, BNP, true, false>(tmA, tmB, tmB1, tmOut, tmRes, grid, K, tiles_n, nsplit, ep, st);
  }
  return launch_tc2_k<MODE, BNP, false, false>(tmA, tmB, tmB1, tmOut, tmRes, grid, K, tiles_n, nsplit, ep, st);
}

// Deferred split-K plan for a residual GEMM whose consumer is a LayerNorm (the FFN w_2 projections, K = 3072):
// with one 256 x 128 pair-tile per cluster only 84 SMs work and each ingests K * 384 * 2 bytes; slicing K over
// `nsplit` clusters per (wider) pair-tile puts <= 74 clusters in one wave with 1/nsplit of the k-blocks each.
// 256-wide pair-tiles x 3 slices beat 384 wide and 2 or 4 slices (profiles/r02_variants_ab.txt).
// Returns 0 (no plan) or fills nsplit.
constexpr int kSplitPairTile = 256;
int gemm_tc2_splitk_plan(int M, int N, int K, int* nsplit) {
  constexpr int ws = kW2Splits;   // the LayerNorm that consumes the slices is instantiated for this count
  if (M < 256 || K % 64 != 0 || N % kSplitPairTile != 0) return 0;
  const int tiles = cdiv(M, 256) * (N / kSplitPairTile);
  if ((K / 64) % ws != 0 || K / 64 / ws < 4 || tiles * ws > 74) return 0;
  *nsplit = ws;
  return 1;
}

// partial[s][M][N] (fp32, s < nsplit) = A[:, slice s of K] * Bw[:, slice s of K]^T -- no bias, no residual
int gemm_tc2_splitk(const void* A, const void* Bw, int M, int N, int K, float* partial, int nsplit, cudaStream_t st) {
  EpiParams ep{};
  ep.M = M; ep.N = N; ep.out = partial; ep.ldo = N;
  AVSR_REQUIRE((reinterpret_cast<uintptr_t>(partial) & 15) == 0, "split-K partial buffer must be 16-byte aligned");
  return launch_tc2<EPI_LINEAR, kSplitPairTile>(reinterpret_cast<const __half*>(A), reinterpret_cast<const __half*>(Bw),
                                                M, N, K, ep, st, nsplit);
}

int gemm_tc2_lse_ok(int M, int N, int K) { return M >= 256 && N % 512 == 0 && K % 64 == 0 && cdiv(M, 256) * (N / 512) <= 74; }

int gemm_tc2_lse(const void* A, const void* Bw, const float* bias, int M, int N, int K, int n_valid, float* logits,
                 long ldo, LsePart* part, int* nparts, cudaStream_t st) {
  AVSR_REQUIRE(gemm_tc2_lse_ok(M, N, K), "gemm_tc2_lse: shape M=%d N=%d K=%d not supported", M, N, K);
  AVSR_REQUIRE(ldo % 4 == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 && n_valid > 0 && n_valid <= N,
               "gemm_tc2_lse: bad output layout");
  EpiParams ep{};
  ep.M = M; ep.N = N; ep.bias = bias; ep.out = logits; ep.ldo = ldo; ep.n_valid = n_valid; ep.lse_part = part;
  *nparts = 2 * (N / 512);
  return launch_tc2<EPI_LSE, 512>(reinterpret_cast<const __half*>(A), reinterpret_cast<const __half*>(Bw), M, N, K, ep, st);
}

// Returns AVSR_OK and sets *handled = 1 when the pair kernel took the GEMM; *handled = 0 -> caller uses gemm_tc.
int gemm_tc2_try(int mode, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st,
                 int* handled) {
  *handled = 0;
  if (K % 64 != 0 || N % 8 != 0 || M < 256) return AVSR_OK;
  if (mode != EPI_LINEAR && mode != EPI_QK && mode != EPI_GLU) return AVSR_OK;
  if (mode == EPI_LINEAR &&
      ((ep.ldo % 8) != 0 || (reinterpret_cast<uintptr_t>(ep.out) & 15) || (reinterpret_cast<uintptr_t>(ep.resid) & 15)))
    return AVSR_OK;
  if (mode == EPI_GLU && ((ep.ldo % 4) != 0 || N % 128 != 0)) return AVSR_OK;
  if (mode == EPI_QK && (N % 128 != 0 || (ep.H * kHeadDim) % 64 != 0)) return AVSR_OK;
  // Pair-tile width: per-SM ingest ~ (128 + BNP/2) * K * 2 bytes shrinks with BNP, so take the NARROWEST width whose
  // pair-tiles still fit one wave of 74 clusters (a second wave would double the time of this one-tile-per-cluster
  // kernel): FFN w_1 (N = 3072) -> 384 (56 pairs), FFN w_2 / out / pw2 (N = 768) -> 128 (42 pairs), QKV (N = 2304)
  // -> 256 (63 pairs), pw1+GLU (N = 1536) -> 256 (42 pairs; GLU needs whole 128-column groups).
  const int tiles_m = cdiv(M, 256);
  int bnp = 0;
  // (a 256 x 96 tile -- 56 clusters for N = 768 -- was measured slower than 256 x 128: 1.862 vs 1.838 ms per forward)
  for (int cand : {128, 256, 384, 512}) {
    if (mode == EPI_GLU && cand < 128) continue;
    if (mode != EPI_LINEAR && cand > 256) continue;            // QK / GLU instantiated for 128 and 256 only
    if (N % cand == 0 && tiles_m * (N / cand) <= 74) { bnp = cand; break; }
  }
  if (!bnp) return AVSR_OK;
  if (mode == EPI_LINEAR && ep.resid && bnp != 128) return AVSR_OK;   // the residual epilogue exists for 256x128 tiles
  *handled = 1;
  const __half* a = reinterpret_cast<const __half*>(A);
  const __half* b = reinterpret_cast<const __half*>(Bw);
  if (mode == EPI_QK) return bnp == 256 ? launch_tc2<EPI_QK, 256>(a, b, M, N, K, ep, st) : launch_tc2<EPI_QK, 128>(a, b, M, N, K, ep, st);
  if (mode == EPI_GLU) return bnp == 256 ? launch_tc2<EPI_GLU, 256>(a, b, M, N, K, ep, st) : launch_tc2<EPI_GLU, 128>(a, b, M, N, K, ep, st);
  if (bnp == 512) return launch_tc2<EPI_LINEAR, 512>(a, b, M, N, K, ep, st);
  if (bnp == 384) return launch_tc2<EPI_LINEAR, 384>(a, b, M, N, K, ep, st);
  if (bnp == 256) return launch_tc2<EPI_LINEAR, 256>(a, b, M, N, K, ep, st);
  return launch_tc2<EPI_LINEAR, 128>(a, b, M, N, K, ep, st);
}

}  // namespace avsr
