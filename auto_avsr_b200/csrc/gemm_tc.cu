// Tensor-core GEMM for the Conformer layer's projections (FFN x2, QK, V^T, out, pw1+GLU, pw2) and the stacked
// linear_pos:   acc[m][n] = sum_k A[m][k] * Bw[n][k]   (both K-major = torch.nn.Linear layout).
//
// Blackwell-native pipeline (sm_100a).  One CTA owns a (MSUB*128) x BN output tile:
//   warp 0   : TMA producer  -- cp.async.bulk.tensor 2-D boxes (rows x 128 bytes, SWIZZLE_128B) of A (MSUB boxes) and
//                               Bw into a STAGES-deep shared-memory ring, completion on `full` mbarriers
//   warp 1   : MMA issuer    -- one thread issues tcgen05.mma (M=128, N=BN, K=32 bytes) x4 x MSUB per stage straight
//                               from shared memory into MSUB TMEM accumulators; tcgen05.commit releases the stage
//                               (`empty` mbarrier) and finally signals `tmem_full`
//   warps 2-9: epilogue      -- tcgen05.ld 32 lanes x 32 columns, fused epilogue (bias / ReLU / residual / GLU /
//                               head-major scatter / conversion to the next operand's storage), direct global stores
// Operand storage (template TOp): float = TF32 (kind::tf32, 8 elements per MMA-K) or __half (kind::f16, 16 per
// MMA-K; same 10-bit mantissa, half the bytes, twice the rate).  Out-of-bounds rows of edge tiles are zero-filled
// by TMA and masked in the epilogue.  With fp32/fp16 operands this GEMM is L2->SM bandwidth bound at M = 1600
// rows, so the tile shape is chosen per problem by a small cost model (bytes through L2 vs tensor-pipe time).
#include "common.cuh"
#include "epilogue.cuh"
#include "sm100.cuh"

namespace avsr {

using namespace sm100;

// ---------------------------------------------------------------- host: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

int make_tmap_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows,
                 int esz) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return AVSR_E_CUDA; }
  AVSR_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld * esz) % 16 == 0 && box_rows <= 256 &&
                   (esz == 4 || esz == 2),
               "tensor map: base/stride must be 16-byte aligned (ld=%llu, esz=%d)", (unsigned long long)ld, esz);
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstr[1] = {ld * (uint64_t)esz};
  cuuint32_t box[2] = {(cuuint32_t)(128 / esz), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, esz == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                   const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(2d) failed: CUresult %d", (int)r); return AVSR_E_CUDA; }
  return AVSR_OK;
}

int make_tmap_3d(CUtensorMap* map, const void* base, uint64_t planes, uint64_t rows, uint64_t cols, uint64_t ld_row,
                 uint64_t ld_plane, uint32_t box_rows, int esz) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) { set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)"); return AVSR_E_CUDA; }
  AVSR_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld_row * esz) % 16 == 0 &&
                   (ld_plane * esz) % 16 == 0 && box_rows <= 256 && (esz == 4 || esz == 2),
               "tensor map 3d: base/strides must be 16-byte aligned");
  cuuint64_t gdim[3] = {cols, rows, planes};
  cuuint64_t gstr[2] = {ld_row * (uint64_t)esz, ld_plane * (uint64_t)esz};
  cuuint32_t box[3] = {(cuuint32_t)(128 / esz), box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, esz == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                   const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(3d) failed: CUresult %d", (int)r); return AVSR_E_CUDA; }
  return AVSR_OK;
}

// ---------------------------------------------------------------- the kernel
constexpr int TC_BM = 128;          // rows per UMMA / per A box
constexpr int TC_THREADS = 320;     // TMA warp + MMA warp + 8 epilogue warps
constexpr int TC_SMEM_BUDGET = 222 * 1024;   // one persistent CTA per SM

template <int BN, int MSUB>
struct TcCfg {
  static constexpr int kABytes = MSUB * TC_BM * 128;
  static constexpr int kBBytes = BN * 128;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kAccStages = (2 * MSUB * BN <= 512) ? 2 : 1;   // double-buffered accumulator when it fits TMEM
  static constexpr int kTmemCols = kAccStages * MSUB * BN;
  static constexpr int kVecBytes = 3 * BN * 4;          // bias / pos_bias_u / pos_bias_v of the tile's columns
  static constexpr int kStagingBytes = 8 * STG_WARP;    // epilogue transpose buffers (dedicated: the ring stays busy)
  static constexpr int kFixedBytes = 1024 /*align slack*/ + 256 /*barriers*/ + kVecBytes + kStagingBytes;
  static constexpr int kStagesFit = (TC_SMEM_BUDGET - kFixedBytes) / kStageBytes;
  static constexpr int kStages = kStagesFit > 8 ? 8 : kStagesFit;
  static constexpr int kSmem = kStages * kStageBytes + kFixedBytes;
  static_assert(kStages >= 2, "tile too large for shared memory");
  static_assert(kTmemCols <= 512 && (kTmemCols & (kTmemCols - 1)) == 0, "TMEM columns must be a power of two <= 512");
};

template <typename TOp> struct OpTraits;
template <> struct OpTraits<float> {
  static constexpr int kElemsPerBlock = 32;  // 128 bytes of fp32
  __device__ static uint32_t idesc(int M, int N) { return umma_idesc_tf32(M, N); }
  __device__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) { mma_tf32(d, a, b, id, acc); }
};
template <> struct OpTraits<__half> {
  static constexpr int kElemsPerBlock = 64;  // 128 bytes of fp16
  __device__ static uint32_t idesc(int M, int N) { return umma_idesc_f16(M, N); }
  __device__ static void mma(uint32_t d, uint64_t a, uint64_t b, uint32_t id, uint32_t acc) { mma_f16(d, a, b, id, acc); }
};

template <int MODE, int BN, int MSUB, typename TOp>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int K, int tiles_m,
               int tiles_n, EpiParams ep) {
  // PERSISTENT: CTA c processes tiles c, c + gridDim.x, ... (n fastest, so concurrently running CTAs share A rows in
  // L2).  The TMA ring never drains between tiles and the accumulator is double-buffered in TMEM, so the epilogue of
  // tile i overlaps the main loop of tile i+1 (at K = 768 a tile is only 12 k-blocks: per-tile prologue / pipeline
  // fill / drain latency was ~3x the tensor-pipe time in the one-tile-per-CTA version, r01 tile sweep).
  using Cfg = TcCfg<BN, MSUB>;
  using Op = OpTraits<TOp>;
  constexpr int S = Cfg::kStages;
  constexpr int ACC = Cfg::kAccStages;
  constexpr int KE = Op::kElemsPerBlock;
  extern __shared__ uint8_t tc_smem_raw[];
  const uint32_t raw = smem_u32(tc_smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;       // SWIZZLE_128B tiles need 1024-byte alignment
  uint8_t* gen = tc_smem_raw + (base - raw);
  const uint32_t bars = base + S * Cfg::kStageBytes;  // full[S], empty[S], tmem_full[2], tmem_empty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gen + S * Cfg::kStageBytes + (2 * S + 4) * 8);
  float* s_vec = reinterpret_cast<float*>(gen + S * Cfg::kStageBytes + 256);   // [3][BN]
  uint8_t* stg_base = gen + S * Cfg::kStageBytes + 256 + Cfg::kVecBytes;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (S + s); };
  auto tmem_full_bar = [&](int a) { return bars + 8u * (2 * S + a); };
  auto tmem_empty_bar = [&](int a) { return bars + 8u * (2 * S + 2 + a); };

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nkb = K / KE;
  const int total_tiles = tiles_m * tiles_n;

  pdl_launch_dependents();
  AVSR_TSPAN_OPEN(400 + MODE, (unsigned)BN | ((unsigned)MSUB << 16));
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < S; ++s) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(tmem_full_bar(a), 1); mbar_init(tmem_empty_bar(a), 8); }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::kTmemCols>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // everything above overlapped the previous kernel's tail; from here on we touch its outputs
  AVSR_TSPAN_DEP();

  // producer / MMA warps: warp-uniform loops, only the instruction issue is guarded by elect.sync (operands stay in
  // uniform registers; see sm100.cuh elect_one_sync)
  if (warp == 0) {
    {
      int it = 0;                                       // running k-block counter across tiles
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int m0 = (tile / tiles_n) * (TC_BM * MSUB), n0 = (tile % tiles_n) * BN;
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          mbar_wait(empty_bar(s), ph ^ 1);
          if (elect_one_sync()) {
            mbar_expect_tx(full_bar(s), Cfg::kStageBytes);
            const uint32_t a_dst = base + s * Cfg::kStageBytes;
#pragma unroll
            for (int ms = 0; ms < MSUB; ++ms)
              tma_load_2d(a_dst + ms * (TC_BM * 128), &tmA, kb * KE, m0 + ms * TC_BM, full_bar(s));
            tma_load_2d(a_dst + Cfg::kABytes, &tmB, kb * KE, n0, full_bar(s));
          }
        }
      }
    }
  } else if (warp == 1) {
    {
      const uint32_t idesc = Op::idesc(TC_BM, BN);
      int it = 0, t = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++t) {
        const int acc = (ACC == 2) ? (t & 1) : 0;
        const uint32_t acc_ph = ((ACC == 2) ? (t >> 1) : t) & 1;
        mbar_wait(tmem_empty_bar(acc), acc_ph ^ 1);     // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * (MSUB * BN);
        for (int kb = 0; kb < nkb; ++kb, ++it) {
          const int s = it % S;
          const uint32_t ph = (it / S) & 1;
          mbar_wait(full_bar(s), ph);
          tc_fence_after();
          const uint32_t a_addr = base + s * Cfg::kStageBytes;
          const uint64_t b_desc = umma_desc_sw128(a_addr + Cfg::kABytes);
          if (elect_one_sync()) {
#pragma unroll
            for (int ms = 0; ms < MSUB; ++ms) {
              const uint64_t a_desc = umma_desc_sw128(a_addr + ms * (TC_BM * 128));
#pragma unroll
              for (int k = 0; k < 4; ++k)  // one MMA-K = 32 bytes = +2 in the descriptor's 16-byte address field
                Op::mma(tacc + ms * BN, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb != 0) || (k != 0));
            }
            tc_commit(empty_bar(s));
            if (kb == nkb - 1) tc_commit(tmem_full_bar(acc));
          }
        }
      }
    }
  } else {
    const int q = warp & 3;                      // TMEM lane quarter this warp may read
    const int chalf = (warp - 2) >> 2;           // which half of the tile's columns this warp drains
    uint8_t* stg = stg_base + (warp - 2) * STG_WARP;
    const int cb = chalf * (BN / 2), ce = cb + BN / 2;      // this warp's columns of the tile
    const int pr = lane >> 3;                                // row (of 4) this lane emits per read iteration
    const int pc = lane & 7;                                 // 16-byte piece of the 128-byte row segment
    constexpr int OC = StageOp<TOp>::kCols;                  // operand columns per row segment (32 tf32 / 64 f16)
    constexpr int ONE = 16 / (int)sizeof(TOp);               // operand elements per 16-byte piece
    int t = 0;
#pragma unroll 1
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++t) {
    const int m0 = (tile / tiles_n) * (TC_BM * MSUB), n0 = (tile % tiles_n) * BN;
    const int acc = (ACC == 2) ? (t & 1) : 0;
    const uint32_t acc_ph = ((ACC == 2) ? (t >> 1) : t) & 1;
    // stage the tile's per-column vectors in shared memory (overlaps the main loop of this tile)
    {
      float* s_bias = s_vec;
      float* s_u = s_vec + BN;
      float* s_v = s_vec + 2 * BN;
      const int D = ep.H * kHeadDim;
      asm volatile("bar.sync 1, 256;" ::: "memory");   // previous tile's readers of s_vec are done
      for (int c = threadIdx.x - 64; c < BN; c += TC_THREADS - 64) {
        const int n = n0 + c;
        float bv = 0.f, uv = 0.f, vv = 0.f;
        if constexpr (MODE != EPI_VT && MODE != EPI_POS) {
          if (ep.bias && n < ep.N) bv = ep.bias[n];
        }
        if constexpr (MODE == EPI_QK) {
          if (n < D) { uv = ep.pos_u[n]; vv = ep.pos_v[n]; }
        }
        s_bias[c] = bv; s_u[c] = uv; s_v[c] = vv;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");   // the 8 epilogue warps only
    }
    mbar_wait(tmem_full_bar(acc), acc_ph);
    tc_fence_after();
    const uint32_t tacc = tmem_base + acc * (MSUB * BN);
#pragma unroll 1
    for (int ms = 0; ms < MSUB; ++ms) {
      const int mw = m0 + ms * TC_BM + q * 32;               // first row of this warp's 32-row slab
      const uint32_t trow = tacc + ((uint32_t)(q * 32) << 16) + ms * BN;
      if constexpr (MODE == EPI_GLU) {
        static_assert(MODE != EPI_GLU || BN % 128 == 0, "GLU pairs live 64 columns apart inside a 128-wide group");
#pragma unroll 1
        for (int g = 0; g < BN; g += 128) {
          const int c = g + chalf * 32;
          float val[32], gate[32];
          tmem_ld32(trow + c, val);
          tmem_ld32(trow + c + 64, gate);
          tmem_ld_wait();
          const float* sb = s_vec + c;
#pragma unroll
          for (int j = 0; j < 32; ++j) val[j] = (val[j] + sb[j]) * sigmoidf_fast(gate[j] + sb[64 + j]);
          stage_write_f32(stg, lane, val, false);
          __syncwarp();
#pragma unroll
          for (int it = 0; it < 8; ++it) emit_glu(ep, mw + it * 4 + pr, n0 + c + pc * 4, stage_read(stg, it, lane));
          __syncwarp();
        }
      } else if constexpr (MODE == EPI_LINEAR) {
        if (!ep.round_out) {                                 // fp32 destination (+ residual)
#pragma unroll 1
          for (int c = cb; c < ce; c += 32) {
            float v[32];
            tmem_ld32(trow + c, v);
            tmem_ld_wait();
            const float* sb = s_vec + c;
#pragma unroll
            for (int j = 0; j < 32; ++j) { v[j] += sb[j]; if (ep.relu) v[j] = fmaxf(v[j], 0.f); }
            stage_write_f32(stg, lane, v, false);
            __syncwarp();
            const int n = n0 + c + pc * 4;
            // residual pieces first (8 independent coalesced loads in flight), then combine + store: a load may not
            // be hoisted above a store by the compiler (possible aliasing), so the order is made explicit here
            float4 r[8];
            if (ep.resid) {
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                const int m = mw + it * 4 + pr;
                r[it] = (m < ep.M && n < ep.N) ? *reinterpret_cast<const float4*>(ep.resid + (long)m * ep.ldo + n)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
              }
            }
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const int m = mw + it * 4 + pr;
              const uint4 pay = stage_read(stg, it, lane);
              float4 o = *reinterpret_cast<const float4*>(&pay);
              if (ep.resid) {
                o.x = r[it].x + ep.alpha * o.x; o.y = r[it].y + ep.alpha * o.y;
                o.z = r[it].z + ep.alpha * o.z; o.w = r[it].w + ep.alpha * o.w;
              }
              if (m < ep.M && n < ep.N)
                *reinterpret_cast<float4*>(reinterpret_cast<float*>(ep.out) + (long)m * ep.ldo + n) = o;
            }
            __syncwarp();
          }
        } else {                                             // operand-typed destination (FFN hidden)
#pragma unroll 1
          for (int c = cb; c < ce; c += OC) {
            float v[OC];
#pragma unroll
            for (int k = 0; k < OC; k += 32) tmem_ld32(trow + c + k, v + k);
            tmem_ld_wait();
            const float* sb = s_vec + c;
#pragma unroll
            for (int j = 0; j < OC; ++j) { v[j] += sb[j]; if (ep.relu) v[j] = fmaxf(v[j], 0.f); }
            StageOp<TOp>::write(stg, lane, v);
            __syncwarp();
#pragma unroll
            for (int it = 0; it < 8; ++it)
              emit_linear_op<TOp>(ep, mw + it * 4 + pr, n0 + c + pc * ONE, stage_read(stg, it, lane));
            __syncwarp();
          }
        }
      } else {
        float row_bias = 0.f;                                // V^T: the bias is per output ROW (feature)
        if constexpr (MODE == EPI_VT) { const int m = mw + lane; row_bias = (m < ep.M) ? ep.bias[m] : 0.f; }
        const int D = ep.H * kHeadDim;
#pragma unroll 1
        for (int c = cb; c < ce; c += OC) {
          float v[OC];
#pragma unroll
          for (int k = 0; k < OC; k += 32) tmem_ld32(trow + c + k, v + k);
          tmem_ld_wait();
          const int n = n0 + c;
          if constexpr (MODE == EPI_QK) {
            const float* sb = s_vec + c;
#pragma unroll
            for (int j = 0; j < OC; ++j) v[j] += sb[j];
            // decode once per chunk / per lane: column -> (segment, head, offset); rows -> (utterance, frame)
            const int np = n + pc * ONE;
            const int seg = np / D, nn = np - seg * D;
            const int hh = nn >> 6, d0 = nn & 63;
            int rb[8], rt[8];
            bool rok[8];
            {
              const int mrow = mw + pr;                    // this lane's first row; the others follow 4 rows apart
              int bb = mrow / ep.T, tt = mrow - bb * ep.T;
#pragma unroll
              for (int it = 0; it < 8; ++it) {
                rb[it] = bb; rt[it] = tt; rok[it] = (mrow + it * 4 < ep.M) && (np < ep.N);
                tt += 4;
                while (tt >= ep.T) { tt -= ep.T; ++bb; }
              }
            }
            if (n < D) {                                     // q: two outputs, q + pos_bias_u and q + pos_bias_v
              const float* su = s_vec + BN + c;
#pragma unroll
              for (int j = 0; j < OC; ++j) v[j] += su[j];
              StageOp<TOp>::write(stg, lane, v);
              __syncwarp();
#pragma unroll
              for (int it = 0; it < 8; ++it)
                emit_heads<TOp>(ep, ep.qu, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
              __syncwarp();
              // second output: re-read the accumulator chunk (cheaper than keeping two register copies)
#pragma unroll
              for (int k = 0; k < OC; k += 32) tmem_ld32(trow + c + k, v + k);
              tmem_ld_wait();
              const float* sv = s_vec + 2 * BN + c;
#pragma unroll
              for (int j = 0; j < OC; ++j) v[j] += sb[j] + sv[j];
              StageOp<TOp>::write(stg, lane, v);
              __syncwarp();
#pragma unroll
              for (int it = 0; it < 8; ++it)
                emit_heads<TOp>(ep, ep.qv, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
              __syncwarp();
            } else {
              StageOp<TOp>::write(stg, lane, v);
              __syncwarp();
              void* dst = n < 2 * D ? ep.kk : ep.vt;
#pragma unroll
              for (int it = 0; it < 8; ++it)
                emit_heads<TOp>(ep, dst, rok[it], rb[it], rt[it], hh, d0, stage_read(stg, it, lane));
              __syncwarp();
            }
          } else {
            if constexpr (MODE == EPI_VT) {
#pragma unroll
              for (int j = 0; j < OC; ++j) v[j] += row_bias;
            }
            StageOp<TOp>::write(stg, lane, v);
            __syncwarp();
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              const uint4 pay = stage_read(stg, it, lane);
              if constexpr (MODE == EPI_VT) emit_vt<TOp>(ep, mw + it * 4 + pr, n + pc * ONE, pay);
              else emit_pos<TOp>(ep, mw + it * 4 + pr, n + pc * ONE, pay);
            }
            __syncwarp();
          }
        }
      }
    }
    // this warp's tcgen05.ld of the accumulator are complete: hand it back to the MMA issuer
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tmem_empty_bar(acc));
    }  // tile loop
  }
  tc_fence_before();
  __syncthreads();
  AVSR_TSPAN_CLOSE();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

AVSR_TRACE_DEFINE_BIND(trace_bind_gemm_tc)

static int num_sms() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

template <int MODE, int BN, int MSUB, typename TOp>
static int launch_tc(const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st) {
  using Cfg = TcCfg<BN, MSUB>;
  CUtensorMap tmA, tmB;
  AVSR_TRY(make_tmap_2d(&tmA, A, (uint64_t)M, (uint64_t)K, (uint64_t)K, TC_BM, (int)sizeof(TOp)));
  AVSR_TRY(make_tmap_2d(&tmB, Bw, (uint64_t)N, (uint64_t)K, (uint64_t)K, BN, (int)sizeof(TOp)));
  AVSR_SET_MAX_SMEM((gemm_tc_kernel<MODE, BN, MSUB, TOp>), Cfg::kSmem);
  const int tiles_m = cdiv(M, TC_BM * MSUB), tiles_n = cdiv(N, BN);
  const int total = tiles_m * tiles_n;
  const int grid = total < num_sms() ? total : num_sms();
  AVSR_LAUNCH((gemm_tc_kernel<MODE, BN, MSUB, TOp>), grid, TC_THREADS, Cfg::kSmem, st, tmA, tmB, K, tiles_m, tiles_n, ep);
  return AVSR_OK;
}

// ---------------------------------------------------------------- tile selection
// Cost model (SM cycles) of one GEMM on 148 persistent CTAs.  What the r01 profiles showed: an SM ingests only
// ~46 B/cycle through TMA (B300_MICROARCH "TMA service/SM"; measured 32 KB per ~690 cycles), well below what the
// tensor pipe consumes, so time ~ (bytes pulled by the busiest SM) / 46 unless the tensor pipe is slower; the
// epilogue hides behind the next tile when the accumulator is double-buffered.  (A deterministic split-K over the
// residual-stream GEMMs was measured slower at S2, 2.45 vs 2.26 ms per forward: its fix-up re-reads the fp32
// partial tiles through the same port as a serial tail.  It was removed; git history has it.)
struct TileChoice { int bn, msub; };
static const int kTileShapes[][2] = {{64, 1}, {128, 1}, {128, 2}, {256, 1}, {256, 2}};

static TileChoice choose_tile(int mode, int M, int N, int K, int esz, bool operand_dest) {
  const double mac_per_cycle = esz == 2 ? 4096.0 : 2048.0;   // per SM, dense f16 / tf32
  const double ingest = 46.0;                                // TMA bytes per cycle per SM
  const int nkb = K / (128 / esz);
  const int sms = 148;
  double best = 1e30;
  TileChoice pick{128, 1};
  for (const auto& sh : kTileShapes) {
    const int bn = sh[0], msub = sh[1];
    if (mode == EPI_GLU && bn % 128 != 0) continue;
    if (bn == 64 && esz == 2 && (mode != EPI_LINEAR || operand_dest)) continue;   // needs 64-column row segments
    if (bn > 64 && N <= bn / 2) continue;                                          // mostly empty tile
    const long tiles = (long)cdiv(M, 128 * msub) * cdiv(N, bn);
    const long per_sm = (tiles + sms - 1) / sms;
    const double kfrac = (double)nkb * (128 / esz);                               // K elements of a tile
    const double t_mma = per_sm * (double)msub * 128.0 * bn * kfrac / mac_per_cycle;
    const double t_in = per_sm * ((double)msub * 128 + bn) * kfrac * esz / ingest;
    const bool acc2 = 2 * msub * bn <= 512;
    const double drain = (double)msub * bn * 10.0;                                 // one tile's epilogue
    const double t_epi = acc2 ? drain : per_sm * drain;
    const double est = (t_mma > t_in ? t_mma : t_in) + t_epi + 4000.0;
    if (est < best) { best = est; pick = TileChoice{bn, msub}; }
  }
  return pick;
}

template <int MODE, typename TOp>
static int dispatch_tile(TileChoice t, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep,
                         cudaStream_t st) {
  if (t.bn == 64) {
    if constexpr (MODE != EPI_GLU) return launch_tc<MODE, 64, 1, TOp>(A, Bw, M, N, K, ep, st);
  }
  if (t.bn == 128 && t.msub == 1) return launch_tc<MODE, 128, 1, TOp>(A, Bw, M, N, K, ep, st);
  if (t.bn == 128 && t.msub == 2) return launch_tc<MODE, 128, 2, TOp>(A, Bw, M, N, K, ep, st);
  if (t.bn == 256 && t.msub == 1) return launch_tc<MODE, 256, 1, TOp>(A, Bw, M, N, K, ep, st);
  if (t.bn == 256 && t.msub == 2) return launch_tc<MODE, 256, 2, TOp>(A, Bw, M, N, K, ep, st);
  set_error("gemm_tc: no kernel for tile %dx%d", t.msub * 128, t.bn);
  return AVSR_E_INVALID;
}

template <typename TOp>
static int dispatch_mode(int mode, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep,
                         cudaStream_t st) {
  const bool operand_dest = mode != EPI_GLU && (mode != EPI_LINEAR || ep.round_out != 0);
  const TileChoice t = choose_tile(mode, M, N, K, (int)sizeof(TOp), operand_dest);
  AVSR_REQUIRE(mode == EPI_VT || N % 8 == 0, "gemm_tc: N=%d must be a multiple of 8", N);
  if (mode == EPI_LINEAR) {
    AVSR_REQUIRE((ep.ldo % 8) == 0 && (reinterpret_cast<uintptr_t>(ep.out) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(ep.resid) & 15) == 0,
                 "gemm_tc: output / residual must be 16-byte aligned with a row stride that is a multiple of 8");
  }
  switch (mode) {
    case EPI_LINEAR: return dispatch_tile<EPI_LINEAR, TOp>(t, A, Bw, M, N, K, ep, st);
    case EPI_QK:
      AVSR_REQUIRE(N % 128 == 0, "gemm_tc: QK needs N %% 128 == 0 (N=%d)", N);
      return dispatch_tile<EPI_QK, TOp>(t, A, Bw, M, N, K, ep, st);
    case EPI_VT:
      AVSR_REQUIRE(M % 64 == 0, "gemm_tc: V^T needs M %% 64 == 0 (M=%d)", M);
      return dispatch_tile<EPI_VT, TOp>(t, A, Bw, M, N, K, ep, st);
    case EPI_GLU:
      AVSR_REQUIRE(N % 128 == 0, "gemm_tc: GLU needs N %% 128 == 0 (N=%d)", N);
      return dispatch_tile<EPI_GLU, TOp>(t, A, Bw, M, N, K, ep, st);
    case EPI_POS:
      AVSR_REQUIRE(N % 64 == 0, "gemm_tc: POS needs N %% 64 == 0 (N=%d)", N);
      return dispatch_tile<EPI_POS, TOp>(t, A, Bw, M, N, K, ep, st);
    default:
      AVSR_REQUIRE(false, "gemm_tc: bad epilogue mode %d", mode);
  }
  return AVSR_OK;
}

int gemm_tc(int mode, int opk, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep,
            cudaStream_t st) {
  AVSR_REQUIRE(opk == OP_TF32 || opk == OP_F16, "gemm_tc: operand kind %d", opk);
  const int ke = opk == OP_F16 ? 64 : 32;
  AVSR_REQUIRE(K >= ke && K % ke == 0, "gemm_tc: K=%d must be a multiple of %d", K, ke);
  if (M <= 0 || N <= 0) return AVSR_OK;
  if (opk == OP_F16) {      // CTA-pair kernel when the problem fits one wave of clusters (half the bytes per MAC per SM)
    int handled = 0;
    AVSR_TRY(gemm_tc2_try(mode, A, Bw, M, N, K, ep, st, &handled));
    if (handled) return AVSR_OK;
  }
  if (opk == OP_F16) return dispatch_mode<__half>(mode, A, Bw, M, N, K, ep, st);
  return dispatch_mode<float>(mode, A, Bw, M, N, K, ep, st);
}

}  // namespace avsr
