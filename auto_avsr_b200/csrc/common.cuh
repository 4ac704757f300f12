// Shared internals of libavsr_b200: error plumbing, launch accounting, the GEMM epilogue family.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <cstdlib>
#include <string>
#include <tuple>
#include <utility>

#include "../../include/avsr_b200.h"

namespace avsr {

// ---------------------------------------------------------------- errors / accounting
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

#define AVSR_CUDA_TRY(expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      ::avsr::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return AVSR_E_CUDA;                                                                     \
    }                                                                                         \
  } while (0)

#define AVSR_CHECK_LAUNCH()                      \
  do {                                           \
    ::avsr::g_launches.fetch_add(1);             \
    AVSR_CUDA_TRY(cudaPeekAtLastError());        \
  } while (0)

#define AVSR_REQUIRE(cond, ...)                  \
  do {                                           \
    if (!(cond)) {                               \
      ::avsr::set_error(__VA_ARGS__);            \
      return AVSR_E_INVALID;                     \
    }                                            \
  } while (0)

#define AVSR_TRY(expr)            \
  do {                            \
    int _r = (expr);              \
    if (_r != AVSR_OK) return _r; \
  } while (0)

constexpr int kHeadDim = 64;  // d_k of the reference encoder (768 / 12); the attention kernels are built for it

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------- programmatic dependent launch (PDL)
// Every hot-path kernel is launched with cudaLaunchAttributeProgrammaticStreamSerialization: it may start (block
// scheduling, barrier init, TMEM allocation, tensor-map prefetch) while its predecessor in the stream / graph is
// still draining, and blocks in pdl_wait() until the predecessor has completed and flushed before it touches any
// global memory.  pdl_launch_dependents() at the top lets the successor do the same.  Without the attribute both
// are no-ops, so the same kernels also work under plain <<<>>> launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args, size_t... I>
inline cudaError_t launch_kernel_impl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                      std::index_sequence<I...>, Args&&... args) {
  std::tuple<KArgs...> params(static_cast<KArgs>(args)...);
  void* ptrs[] = {const_cast<void*>(static_cast<const void*>(&std::get<I>(params)))...};
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelExC(&cfg, reinterpret_cast<const void*>(kernel), ptrs);
}
// launch `kernel<<<grid, block, smem, st>>>(args...)` with the PDL attribute
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
  static_assert(sizeof...(KArgs) == sizeof...(Args), "kernel argument count mismatch");
  return launch_kernel_impl(kernel, grid, block, smem, st, std::index_sequence_for<KArgs...>{}, std::forward<Args>(args)...);
}

// opt a kernel into > 48 KB of dynamic shared memory; remembered per device (one process may drive several GPUs)
#define AVSR_SET_MAX_SMEM(kernel, bytes)                                                                     \
  do {                                                                                                       \
    static int _done_dev = -1;                                                                               \
    int _dev = 0;                                                                                            \
    AVSR_CUDA_TRY(cudaGetDevice(&_dev));                                                                     \
    if (_done_dev != _dev) {                                                                                 \
      AVSR_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))); \
      _done_dev = _dev;                                                                                      \
    }                                                                                                        \
  } while (0)

#define AVSR_LAUNCH(kernel, grid, block, smem, st, ...)                                                \
  do {                                                                                                 \
    ::avsr::g_launches.fetch_add(1);                                                                   \
    AVSR_CUDA_TRY(::avsr::launch_kernel(kernel, dim3(grid), dim3(block), (size_t)(smem), st, __VA_ARGS__)); \
  } while (0)

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float round_tf32(float x) {
  // round-to-nearest (ties away) to the 10-bit TF32 mantissa; the tensor core then truncates nothing.
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return __uint_as_float(r);
}
__device__ __forceinline__ float sigmoidf_acc(float x) { return 1.0f / (1.0f + expf(-x)); }
// sigmoid through ex2.approx + fast reciprocal (relative error ~1e-6: far below the 11-bit operand rounding that
// follows in the tensor-core paths); the fp32 reference path keeps sigmoidf_acc
__device__ __forceinline__ float sigmoidf_fast(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }

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

// ---------------------------------------------------------------- tensor-core operand storage
// How a tensor that feeds a tensor-core contraction is stored:
//   OP_F32  : plain fp32 (CUDA-core reference path)
//   OP_TF32 : fp32 container, value rounded to TF32 (10-bit mantissa) -> tcgen05 kind::tf32
//   OP_F16  : IEEE half (same 10-bit mantissa as TF32, 5-bit exponent, saturating) -> tcgen05 kind::f16;
//             half the bytes through L2/shared memory and twice the MMA rate of kind::tf32
enum OperandKind : int { OP_F32 = 0, OP_TF32 = 1, OP_F16 = 2 };

__device__ __forceinline__ __half to_half_sat(float x) {
  unsigned short r;
  asm("cvt.rn.satfinite.f16.f32 %0, %1;" : "=h"(r) : "f"(x));
  return __ushort_as_half(r);
}
// two floats -> packed IEEE halves (a in the low half), round to nearest, saturating: ONE conversion instruction
__device__ __forceinline__ uint32_t pack_half2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// the same with ReLU folded into the conversion (F2FP.SATFINITE.RELU): negative -> +0, NaN stays NaN like torch.relu
__device__ __forceinline__ uint32_t pack_half2_sat_relu(float a, float b) {
  uint32_t r;
  asm("cvt.rn.relu.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}
// store 4 consecutive operand values (dst 16-byte aligned for float, 8-byte aligned for half)
template <typename TOp>
__device__ __forceinline__ void store_op4(TOp* dst, float a, float b, float c, float d);
template <>
__device__ __forceinline__ void store_op4<float>(float* dst, float a, float b, float c, float d) {
  *reinterpret_cast<float4*>(dst) = make_float4(round_tf32(a), round_tf32(b), round_tf32(c), round_tf32(d));
}
template <>
__device__ __forceinline__ void store_op4<__half>(__half* dst, float a, float b, float c, float d) {
  __half2 lo = __halves2half2(to_half_sat(a), to_half_sat(b));
  __half2 hi = __halves2half2(to_half_sat(c), to_half_sat(d));
  uint2 v;
  v.x = *reinterpret_cast<uint32_t*>(&lo);
  v.y = *reinterpret_cast<uint32_t*>(&hi);
  *reinterpret_cast<uint2*>(dst) = v;
}
template <typename TOp>
__device__ __forceinline__ void store_op1(TOp* dst, float a);
template <>
__device__ __forceinline__ void store_op1<float>(float* dst, float a) { *dst = round_tf32(a); }
template <>
__device__ __forceinline__ void store_op1<__half>(__half* dst, float a) { *dst = to_half_sat(a); }
// runtime-kind store used by the elementwise kernels (kind is warp-uniform)
__device__ __forceinline__ void store_kind4(void* base, long idx, int kind, float a, float b, float c, float d) {
  if (kind == OP_F16) store_op4<__half>(reinterpret_cast<__half*>(base) + idx, a, b, c, d);
  else if (kind == OP_TF32) store_op4<float>(reinterpret_cast<float*>(base) + idx, a, b, c, d);
  else *reinterpret_cast<float4*>(reinterpret_cast<float*>(base) + idx) = make_float4(a, b, c, d);
}

// ---------------------------------------------------------------- GEMM epilogues
// Every GEMM computes acc[m][n] = sum_k A[m][k] * Bw[n][k]  (both operands K-major, i.e. torch Linear).
enum EpiMode : int {
  EPI_LINEAR = 0,  // y = [resid + alpha *] act(acc + bias[n])                      -> out (M, ldo)
  EPI_QK = 1,      // n <  D: q -> qu = q+bias+pos_u, qv = q+bias+pos_v ; D <= n < 2D: k ; 2D <= n < 3D (when
                   // N == 3D): v into `vt` with the SAME head-major layout   -> (B,H,T,64) each
  EPI_VT = 2,      // A = W_v (m = feature), B = frames (n): v^T                     -> (B,H,64,Tp)
  EPI_GLU = 3,     // interleaved pointwise_cov1: value cols [g*128, +64), gate cols +64 -> out (M, N/2)
  EPI_POS = 4,     // linear_pos of all layers: n = l*D + h*64 + d, m = table row      -> (L,H,Rp,64)
  EPI_LSE = 5      // y = acc + bias[n] as fp32 logits (M, ldo) PLUS per (row, half column tile) log-sum-exp partials over
                   // the columns n < n_valid -- the ctc_lo projection (two-SM kernel only, gemm_tc2_lse)
};

// one log-sum-exp partial: running maximum, sum of exp(x - maximum) and first index of the maximum
struct LsePart {
  float m, s;
  int idx, pad;
};

struct EpiParams {
  int M, N;           // logical extents of acc
  const float* bias;  // LINEAR/QK/GLU: [N]; VT: [M]; may be null (LINEAR, POS)
  void* out;          // LINEAR / GLU / POS destination: fp32, or operand-typed when round_out != 0
  long ldo;           // LINEAR / GLU row stride of out
  const float* resid; // LINEAR: optional residual (same layout as out; may alias out)
  float alpha;        // LINEAR: scale of the residual branch
  int relu;           // LINEAR
  int round_out;      // round the stored value to TF32 (it feeds a tensor-core operand)
  int T, H, Tp, Rp;   // frames per utterance, heads, padded T of v^T, padded rows of the pos table
  const float* pos_u; // QK: [H*64]
  const float* pos_v;
  int n_valid;        // LSE: columns >= n_valid are padding (stored, but excluded from the partials)
  LsePart* lse_part;  // LSE: [2 * tiles_n][M] partials (two epilogue warps per lane quarter split a tile's columns)
  void* qu;           // operand-typed (float for OP_F32/OP_TF32, __half for OP_F16)
  void* qv;
  void* kk;
  void* vt;
};

// ---------------------------------------------------------------- phase trace (diagnostic build only)
// scripts/build_trace.py compiles the library with -DAVSR_TRACE into libavsr_b200_trace.so; the product build does
// not contain any of this.  Buffer layout (64-bit words): [0] = records used, [1] = record capacity, then records of
// kTraceWords words: [0] kernel id, [1] blockIdx.x | aux << 32, [2] SM id, [3] %globaltimer at open,
// [4 + s] = clock64() at phase mark s (s < 10), [14] / [15] = %globaltimer when the dependency resolved / the CTA was done.
// One record per CTA; marks are written by whichever thread reaches the phase.
#ifdef AVSR_TRACE
constexpr int kTraceWords = 16;
// Every translation unit has its own copy of the buffer pointer (no relocatable device code in this build); each
// .cu defines a binder with AVSR_TRACE_DEFINE_BIND and avsr_trace_set (encoder.cu) calls all of them.  The kernels
// read the pointer at run time, so a CUDA graph captured before avsr_trace_set still traces.
static __device__ unsigned long long* d_trace_buf;
#define AVSR_TRACE_DEFINE_BIND(name)                                                         \
  int name(unsigned long long* p) {                                                          \
    return cudaMemcpyToSymbol(::avsr::d_trace_buf, &p, sizeof p) == cudaSuccess ? 0 : 1;     \
  }
__device__ __forceinline__ unsigned long long trace_globaltimer() {
  unsigned long long gt;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
  return gt;
}
__device__ __forceinline__ unsigned long long* trace_open(int kernel_id, unsigned aux) {
  unsigned long long* trace = d_trace_buf;
  if (!trace) return nullptr;
  const unsigned long long r = atomicAdd(trace, 1ULL);
  if (r >= trace[1]) return nullptr;
  unsigned long long* rec = trace + 2 + r * kTraceWords;
  unsigned smid;
  asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
  rec[0] = (unsigned long long)kernel_id;
  rec[1] = (unsigned long long)blockIdx.x | ((unsigned long long)aux << 32);
  rec[2] = smid;
  rec[3] = trace_globaltimer();
  return rec;
}
__device__ __forceinline__ void trace_mark(unsigned long long* rec, int slot) {
  if (rec) rec[4 + slot] = (unsigned long long)clock64();
}
// globaltimer stamps for the launch timeline: slot 10 = dependency resolved (after griddepcontrol.wait), 11 = CTA done
__device__ __forceinline__ void trace_stamp(unsigned long long* rec, int slot) {
  if (rec) rec[4 + slot] = trace_globaltimer();
}
#define AVSR_TRACE_OPEN(slot_ptr, id, aux) do { *(slot_ptr) = ::avsr::trace_open(id, aux); } while (0)
#define AVSR_TRACE_MARK(cond, slot_ptr, s) do { if (cond) ::avsr::trace_mark(*(slot_ptr), s); } while (0)
#define AVSR_TRACE_STAMP(cond, slot_ptr, s) do { if (cond) ::avsr::trace_stamp(*(slot_ptr), s); } while (0)
// simple kernels (no shared slot): thread 0 of the CTA keeps the record pointer in a register
#define AVSR_TSPAN_OPEN(id, aux) unsigned long long* _tsp = threadIdx.x == 0 ? ::avsr::trace_open(id, aux) : nullptr
#define AVSR_TSPAN_DEP() ::avsr::trace_stamp(_tsp, 10)
#define AVSR_TSPAN_CLOSE() ::avsr::trace_stamp(_tsp, 11)
#else
#define AVSR_TRACE_DEFINE_BIND(name)
#define AVSR_TRACE_OPEN(slot_ptr, id, aux) do { } while (0)
#define AVSR_TRACE_MARK(cond, slot_ptr, s) do { } while (0)
#define AVSR_TRACE_STAMP(cond, slot_ptr, s) do { } while (0)
#define AVSR_TSPAN_OPEN(id, aux) do { } while (0)
#define AVSR_TSPAN_DEP() do { } while (0)
#define AVSR_TSPAN_CLOSE() do { } while (0)
#endif

// scalar store of one operand-or-fp32 value: `operand` says the destination is TOp-typed (rounded), else plain fp32
template <typename TOp>
__device__ __forceinline__ void put(void* base, long idx, float v, bool operand) {
  if (operand) store_op1<TOp>(reinterpret_cast<TOp*>(base) + idx, v);
  else reinterpret_cast<float*>(base)[idx] = v;
}

// Scalar (one element) epilogue: used by the CUDA-core GEMM and by the tensor-core kernel's ragged edges.
// TOp = float serves OP_F32 (round_out = 0) and OP_TF32 (round_out = 1); TOp = __half serves OP_F16.
template <int MODE, typename TOp = float>
__device__ __forceinline__ void epi_store(const EpiParams& p, int m, int n, float acc) {
  if (m >= p.M || n >= p.N) return;
  if constexpr (MODE == EPI_LINEAR) {
    float v = acc + (p.bias ? p.bias[n] : 0.0f);
    if (p.relu) v = fmaxf(v, 0.0f);
    if (p.resid) v = p.resid[(long)m * p.ldo + n] + p.alpha * v;
    put<TOp>(p.out, (long)m * p.ldo + n, v, p.round_out != 0);
  } else if constexpr (MODE == EPI_QK) {
    const int D = p.H * kHeadDim;
    const int b = m / p.T, t = m - b * p.T;
    const int seg = n / D, nn = n - seg * D;          // 0: q, 1: k, 2: v (merged QKV projection)
    const int h = nn / kHeadDim, d = nn - h * kHeadDim;
    const long idx = (((long)b * p.H + h) * p.T + t) * kHeadDim + d;
    const float v = acc + p.bias[n];
    if (seg == 0) {
      put<TOp>(p.qu, idx, v + p.pos_u[nn], p.round_out != 0);
      put<TOp>(p.qv, idx, v + p.pos_v[nn], p.round_out != 0);
    } else {
      put<TOp>(seg == 1 ? p.kk : p.vt, idx, v, p.round_out != 0);
    }
  } else if constexpr (MODE == EPI_VT) {
    const int b = n / p.T, t = n - b * p.T;
    const int h = m / kHeadDim, d = m - h * kHeadDim;
    put<TOp>(p.vt, (((long)b * p.H + h) * kHeadDim + d) * p.Tp + t, acc + p.bias[m], p.round_out != 0);
  } else if constexpr (MODE == EPI_POS) {
    const int D = p.H * kHeadDim;
    const int l = n / D, r = n - l * D;
    const int h = r / kHeadDim, d = r - h * kHeadDim;
    put<TOp>(p.out, (((long)l * p.H + h) * p.Rp + m) * kHeadDim + d, acc, p.round_out != 0);
  }
}

// GLU pair: n_val is the interleaved column of the value half, the gate sits 64 columns further.  Output is fp32
// (it feeds the depthwise conv, not a tensor-core operand).
__device__ __forceinline__ void epi_store_glu(const EpiParams& p, int m, int n_val, float acc_val, float acc_gate) {
  if (m >= p.M || n_val + 64 >= p.N) return;
  const float a = acc_val + p.bias[n_val];
  const float g = acc_gate + p.bias[n_val + 64];
  const int c = (n_val >> 7) * 64 + (n_val & 63);
  reinterpret_cast<float*>(p.out)[(long)m * p.ldo + c] = a * sigmoidf_acc(g);
}

// ---------------------------------------------------------------- kernel launchers (defined in the .cu files)
// fp32 CUDA-core GEMM (gemm_simt.cu)
int gemm_simt(int mode, const float* A, const float* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st);
// tcgen05 GEMM (gemm_tc.cu); opk = OP_TF32 (A, Bw are float) or OP_F16 (A, Bw are __half)
int gemm_tc(int mode, int opk, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st);

// two-SM (cta_group::2) GEMM for fp16 EPI_LINEAR / EPI_QK / EPI_GLU (gemm_tc2.cu): *handled = 1 when it took the problem
int gemm_tc2_try(int mode, const void* A, const void* Bw, int M, int N, int K, const EpiParams& ep, cudaStream_t st,
                 int* handled);

// deferred split-K (gemm_tc2.cu): plan returns 1 and fills nsplit (= kW2Splits) when the shape qualifies; the GEMM
// writes partial[s][M][N] (raw fp32 k-slice sums) and the consuming LayerNorm finishes the residual update (LnParts)
constexpr int kW2Splits = 3;
int gemm_tc2_splitk_plan(int M, int N, int K, int* nsplit);
// true while the caller guarantees that B operands are prepared weights no kernel of the stream writes (the encoder
// forward): the two-SM GEMM then fetches weights before griddepcontrol.wait
extern thread_local bool g_tc2_weights_static;
int gemm_tc2_splitk(const void* A, const void* Bw, int M, int N, int K, float* partial, int nsplit, cudaStream_t st);

// ctc_lo (gemm_tc2.cu): logits[M][ldo] = A Bw^T + bias (fp32; N a multiple of 512, padded columns included) and
// part[nparts][M] log-sum-exp partials over the columns < n_valid; *nparts = 2 * N / 512.  Needs M >= 256, K % 64 == 0.
int gemm_tc2_lse(const void* A, const void* Bw, const float* bias, int M, int N, int K, int n_valid, float* logits,
                 long ldo, LsePart* part, int* nparts, cudaStream_t st);
int gemm_tc2_lse_ok(int M, int N, int K);

// Residual update folded into a LayerNorm's load: row = x + alpha * (bias + part[0] + part[1] + ... ) (fixed order,
// so the result does not depend on scheduling); the updated row is written to x_out when that is not already the
// LayerNorm's own fp32 output.
struct LnParts {
  const float* part = nullptr;   // [nparts][rows][d]
  int nparts = 0;
  long stride = 0;               // rows * d
  const float* bias = nullptr;   // [d]
  float alpha = 0.f;
  float* x_out = nullptr;        // optional [rows][d]
};

// elementwise.cu
int launch_embed_scale(const float* xs, float* x, long n, float scale, cudaStream_t st);
// `out_kind` is an OperandKind: how y / pe is stored
int launch_layernorm(const float* x, const float* g, const float* b, void* y, int rows, int d, int out_kind,
                     cudaStream_t st, const LnParts* parts = nullptr);
// y_f32 = LN(x) as fp32 (may alias x) AND y_op = the same values in operand storage (after_norm feeding ctc_lo)
int launch_layernorm_dual(const float* x, const float* g, const float* b, float* y_f32, void* y_op, int rows, int d,
                          int out_kind, cudaStream_t st);
int launch_layernorm2(const float* x, const float* g1, const float* b1, const float* g2, const float* b2, float* y1,
                      void* y2, int rows, int d, int out_kind, cudaStream_t st, const LnParts* parts = nullptr);
int launch_sinusoid(void* pe, int T, int d, int out_kind, cudaStream_t st);
int launch_dwconv_bn_silu(const float* x, const float* wt /*(K,C)*/, const float* scale, const float* shift, void* y,
                          int B, int T, int C, int K, int out_kind, cudaStream_t st);

// head.cu
int launch_lse_finish(const float* logits, long ldx, const LsePart* part, int nparts, int rows, float* y, long ldy,
                      int32_t* best, int n, cudaStream_t st);
int launch_log_softmax_rows(const float* x, long ldx, float* y, long ldy, int32_t* best, int rows, int n, cudaStream_t st);

// attention: q-side tensors (B,H,T,64), vt (B,H,64,Tp), pos (H,Rp,64) for one layer, ctx (B*T, H*64)
int attention_simt(const float* qu, const float* qv, const float* kk, const float* vt, const float* pos,
                   const int32_t* lengths, float* ctx, int B, int T, int H, int Tp, int Rp, int round_out,
                   cudaStream_t st);
int attention_tc(const float* qu, const float* qv, const float* kk, const float* vt, const float* pos,
                 const int32_t* lengths, float* ctx, int B, int T, int H, int Tp, int Rp, int round_out,
                 cudaStream_t st);
// fp16 operands (attention_f16.cu): qu, qv, kk, vv all (B,H,T,64) __half (V in its natural layout); ctx __half
int attention_f16(const __half* qu, const __half* qv, const __half* kk, const __half* vv, const __half* pos,
                  const int32_t* lengths, __half* ctx, int B, int T, int H, int Rp, cudaStream_t st);

}  // namespace avsr
