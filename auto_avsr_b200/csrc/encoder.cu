// Host orchestration + C ABI of libavsr_b200: weight preparation, workspace carving, the 12-layer
// forward schedule (ConformerEncoder.forward, conformer_encoder.py:264-282) and the CUDA-graph plan.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <vector>

#include "common.cuh"

namespace avsr {

// ------------------------------------------------------------------ error / accounting
static thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
}

// ------------------------------------------------------------------ prepared-weight layout
struct LayerPrep {
  float *ffm_w1, *ffm_b1, *ffm_w2, *ffm_b2, *ln_ffm_w, *ln_ffm_b;
  float *qk_w, *qk_b, *v_w, *v_b, *out_w, *out_b, *pos_u, *pos_v, *ln_mha_w, *ln_mha_b;
  float *pw1_w, *pw1_b, *dw_wt, *dw_scale, *dw_shift, *pw2_w, *pw2_b, *ln_conv_w, *ln_conv_b;
  float *ff_w1, *ff_b1, *ff_w2, *ff_b2, *ln_ff_w, *ln_ff_b;
  float *ln_fin_w, *ln_fin_b;
};
struct Prepared {
  std::vector<LayerPrep> layers;
  float *pos_w_all, *after_w, *after_b;
  size_t bytes;
};

struct Carver {
  char* base;
  size_t off = 0;
  float* take(size_t nfloats) {
    float* p = reinterpret_cast<float*>(base + off);
    off += align_up(nfloats * sizeof(float), 256);
    return p;
  }
};

static Prepared layout_prepared(const AvsrEncoderConfig& c, void* base) {
  Prepared P;
  Carver cv{reinterpret_cast<char*>(base)};
  const size_t D = c.d_model, F = c.linear_units, K = c.cnn_kernel;
  P.layers.resize(c.num_blocks);
  for (auto& L : P.layers) {
    L.ffm_w1 = cv.take(F * D); L.ffm_b1 = cv.take(F); L.ffm_w2 = cv.take(D * F); L.ffm_b2 = cv.take(D);
    L.ln_ffm_w = cv.take(D); L.ln_ffm_b = cv.take(D);
    L.qk_w = cv.take(3 * D * D); L.qk_b = cv.take(3 * D);   // q | k | v rows contiguous (one QKV GEMM in F16 mode)
    L.v_w = nullptr; L.v_b = L.qk_b + 2 * D;                // v_w is an operand-sized offset into qk_w (see v_weights())
    L.out_w = cv.take(D * D); L.out_b = cv.take(D); L.pos_u = cv.take(D); L.pos_v = cv.take(D);
    L.ln_mha_w = cv.take(D); L.ln_mha_b = cv.take(D);
    L.pw1_w = cv.take(2 * D * D); L.pw1_b = cv.take(2 * D); L.dw_wt = cv.take(K * D);
    L.dw_scale = cv.take(D); L.dw_shift = cv.take(D); L.pw2_w = cv.take(D * D); L.pw2_b = cv.take(D);
    L.ln_conv_w = cv.take(D); L.ln_conv_b = cv.take(D);
    L.ff_w1 = cv.take(F * D); L.ff_b1 = cv.take(F); L.ff_w2 = cv.take(D * F); L.ff_b2 = cv.take(D);
    L.ln_ff_w = cv.take(D); L.ln_ff_b = cv.take(D);
    L.ln_fin_w = cv.take(D); L.ln_fin_b = cv.take(D);
  }
  P.pos_w_all = cv.take((size_t)c.num_blocks * D * D);
  P.after_w = cv.take(D);
  P.after_b = cv.take(D);
  P.bytes = cv.off;
  return P;
}

static int check_cfg(const AvsrEncoderConfig* c) {
  AVSR_REQUIRE(c != nullptr, "config is NULL");
  AVSR_REQUIRE(c->n_heads > 0 && c->d_model == c->n_heads * kHeadDim,
               "d_model=%d must be n_heads=%d * 64 (the attention kernels are built for d_k = 64)", c->d_model,
               c->n_heads);
  AVSR_REQUIRE(c->d_model % 64 == 0 && c->d_model <= 1024, "d_model=%d must be a multiple of 64 and <= 1024", c->d_model);
  AVSR_REQUIRE(c->linear_units > 0 && c->linear_units % 64 == 0, "linear_units=%d must be a multiple of 64",
               c->linear_units);
  AVSR_REQUIRE(c->num_blocks > 0, "num_blocks=%d", c->num_blocks);
  AVSR_REQUIRE(c->cnn_kernel % 2 == 1 && c->cnn_kernel >= 1 && c->cnn_kernel <= 255, "cnn_kernel=%d must be odd",
               c->cnn_kernel);
  return AVSR_OK;
}

// ------------------------------------------------------------------ preparation kernels
// copy with conversion to an operand storage kind (OP_F32 plain copy, OP_TF32 rounded fp32, OP_F16 half)
__global__ void copy_round_kernel(const float* __restrict__ src, void* __restrict__ dst, long n, int kind, float scale) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    const float v = src[i] * scale;
    if (kind == OP_F16) reinterpret_cast<__half*>(dst)[i] = to_half_sat(v);
    else reinterpret_cast<float*>(dst)[i] = kind == OP_TF32 ? round_tf32(v) : v;
  }
}
// pointwise_cov1 (2D, D[,1]) -> rows interleaved in groups of 64: [g*128, +64) value channels g*64.., then their gates
__global__ void glu_interleave_kernel(const float* __restrict__ w, const float* __restrict__ b, void* __restrict__ wo,
                                      float* __restrict__ bo, int D, int kind) {
  const int r = blockIdx.x;  // destination row in [0, 2D)
  const int g = r >> 7, wi = r & 127;
  const int src = wi < 64 ? g * 64 + wi : D + g * 64 + (wi - 64);
  for (int k = threadIdx.x; k < D; k += blockDim.x) {
    const float v = w[(long)src * D + k];
    if (kind == OP_F16) reinterpret_cast<__half*>(wo)[(long)r * D + k] = to_half_sat(v);
    else reinterpret_cast<float*>(wo)[(long)r * D + k] = kind == OP_TF32 ? round_tf32(v) : v;
  }
  if (threadIdx.x == 0) bo[r] = b[src];
}
// depthwise taps (C,1,K) -> (K,C); BN(eval)+conv bias folded: scale = g/sqrt(var+eps), shift = beta + (b - mean)*scale
__global__ void dw_fold_kernel(const float* __restrict__ w, const float* __restrict__ b, const float* __restrict__ bn_w,
                               const float* __restrict__ bn_b, const float* __restrict__ mean,
                               const float* __restrict__ var, float* __restrict__ wt, float* __restrict__ scale,
                               float* __restrict__ shift, int C, int K) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  for (int k = 0; k < K; ++k) wt[(long)k * C + c] = w[(long)c * K + k];
  const float s = bn_w[c] / sqrtf(var[c] + 1e-5f);
  scale[c] = s;
  shift[c] = bn_b[c] + (b[c] - mean[c]) * s;
}

static int copy_round(const float* src, void* dst, long n, int kind, cudaStream_t st, float scale = 1.0f) {
  if (n <= 0) return AVSR_OK;
  int blocks = (int)((n + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  copy_round_kernel<<<blocks, 256, 0, st>>>(src, dst, n, kind, scale);
  AVSR_CHECK_LAUNCH();
  return AVSR_OK;
}

// ------------------------------------------------------------------ precision -> operand storage
static inline bool valid_precision(int p) { return p == AVSR_PREC_FP32 || p == AVSR_PREC_TF32 || p == AVSR_PREC_F16; }
static inline int operand_kind(int precision) {
  return precision == AVSR_PREC_F16 ? OP_F16 : (precision == AVSR_PREC_TF32 ? OP_TF32 : OP_F32);
}
static inline size_t operand_size(int precision) { return precision == AVSR_PREC_F16 ? 2 : 4; }
// element offset into an operand-typed buffer carved as floats
static inline void* op_offset(void* base, size_t elems, int precision) {
  return reinterpret_cast<char*>(base) + elems * operand_size(precision);
}
static inline const void* op_offset(const void* base, size_t elems, int precision) {
  return reinterpret_cast<const char*>(base) + elems * operand_size(precision);
}

// ------------------------------------------------------------------ workspace
struct Workspace {
  float *x, *xn, *hid, *qu, *qv, *kk, *vt, *ctx, *glu, *dw, *pe, *pos;
  float* splitk;      // [kW2Splits][N][d_model] fp32 k-slices of the deferred FFN w_2 GEMM (gemm_tc2_splitk)
  int32_t* lengths;
  int Tp, Rp;
  size_t bytes;
};

static Workspace layout_workspace(const AvsrEncoderConfig& c, int B, int T, void* base) {
  Workspace W;
  Carver cv{reinterpret_cast<char*>(base)};
  const size_t N = (size_t)B * T, D = c.d_model, F = c.linear_units;
  W.Tp = (T + 7) & ~7;   // v^T rows 16-byte aligned for TMA with 2-byte elements too
  W.Rp = 2 * T - 1;
  W.x = cv.take(N * D); W.xn = cv.take(N * D); W.hid = cv.take(N * F);
  W.qu = cv.take(N * D); W.qv = cv.take(N * D); W.kk = cv.take(N * D);
  W.vt = cv.take((size_t)B * D * W.Tp);
  W.ctx = cv.take(N * D); W.glu = cv.take(N * D); W.dw = cv.take(N * D);
  W.pe = cv.take((size_t)W.Rp * D);
  W.pos = cv.take((size_t)c.num_blocks * W.Rp * D);
  W.splitk = cv.take((size_t)kW2Splits * N * D);
  W.lengths = reinterpret_cast<int32_t*>(cv.take((size_t)B));
  W.bytes = cv.off;
  return W;
}

__global__ void fill_lengths_kernel(int32_t* dst, const int32_t* src, int B, int T) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) dst[i] = src ? src[i] : T;
}

// ------------------------------------------------------------------ saturation check (diagnostic forward)
// fp16 operand stores saturate (cvt.rn.satfinite, common.cuh): a value beyond +-65504 becomes +-65504 silently.  The
// checked forward (avsr_encoder_forward_checked) scans every operand tensor right after its producer and counts the
// elements that sit AT the saturation value (or are NaN): non-zero means the fp16 path left its range for these
// weights / inputs and the caller must fall back to tf32 / fp32 precision -- the drop-in raises (engine.py).
__global__ void count_saturated_kernel(const uint4* __restrict__ p, long n16, unsigned long long* count) {
  unsigned local = 0;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n16; i += (long)gridDim.x * blockDim.x) {
    const uint4 v = p[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      local += ((w[k] & 0x7fffu) >= 0x7bffu) ? 1u : 0u;
      local += (((w[k] >> 16) & 0x7fffu) >= 0x7bffu) ? 1u : 0u;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, (unsigned long long)local);
}
static int count_saturated(const void* halfs, size_t nelems, unsigned long long* count, cudaStream_t st) {
  if (!count || nelems == 0) return AVSR_OK;
  AVSR_REQUIRE(nelems % 8 == 0 && (reinterpret_cast<uintptr_t>(halfs) & 15) == 0, "saturation scan: unaligned buffer");
  int blocks = (int)((nelems / 8 + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  count_saturated_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const uint4*>(halfs), (long)(nelems / 8), count);
  AVSR_CHECK_LAUNCH();
  return AVSR_OK;
}

// ------------------------------------------------------------------ forward schedule
static EpiParams epi_linear(int M, int N, const float* bias, void* out, const float* resid, float alpha, int relu,
                            int round_out) {
  EpiParams e{};
  e.M = M; e.N = N; e.bias = bias; e.out = out; e.ldo = N; e.resid = resid; e.alpha = alpha; e.relu = relu;
  e.round_out = round_out;
  return e;
}

static int run_gemm(int prec, int mode, const void* A, const void* Bw, int M, int N, int K, const EpiParams& e,
                    cudaStream_t st) {
  if (prec == AVSR_PREC_FP32)
    return gemm_simt(mode, reinterpret_cast<const float*>(A), reinterpret_cast<const float*>(Bw), M, N, K, e, st);
  return gemm_tc(mode, operand_kind(prec), A, Bw, M, N, K, e, st);
}

// the part of the forward that only touches workspace buffers (what a plan captures into its graph)
// `aux` (optional): a second stream + two events.  The rel-pos table and the stacked linear_pos GEMM only feed the
// attention kernels, so they are forked onto `aux.stream` and joined right before layer 0's attention; inside a
// captured graph this becomes a parallel branch that overlaps layer 0's macaron FFN (the work is still done every
// forward -- nothing is cached across steps).
struct AuxFork {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};

// pos_emb table and linear_pos of every layer in one GEMM (embedding.py:179-183, attention.py:170)
static int compute_pos(const AvsrEncoderConfig& c, const Prepared& P, const Workspace& W, int T, int prec, cudaStream_t ps) {
  const int D = c.d_model, H = c.n_heads, L = c.num_blocks;
  AVSR_TRY(launch_sinusoid(W.pe, T, D, operand_kind(prec), ps));
  EpiParams e{};
  e.M = W.Rp; e.N = L * D; e.out = W.pos; e.H = H; e.Rp = W.Rp; e.round_out = prec != AVSR_PREC_FP32;
  return run_gemm(prec, EPI_POS, W.pe, P.pos_w_all, W.Rp, L * D, D, e, ps);
}

static int forward_body(const AvsrEncoderConfig& c, const Prepared& P, const Workspace& W, int B, int T,
                        const int32_t* lengths, float* taps, int prec, cudaStream_t st, const AuxFork* aux = nullptr,
                        unsigned long long* sat = nullptr) {
  const int N = B * T, D = c.d_model, F = c.linear_units, H = c.n_heads, L = c.num_blocks;
  const int opk = operand_kind(prec);           // storage of every tensor that feeds a contraction
  const int opr = prec != AVSR_PREC_FP32;       // "destination is operand-typed" flag of the epilogues
  const size_t stage_bytes = (size_t)N * D * sizeof(float);
  if (prec != AVSR_PREC_F16) sat = nullptr;     // only the fp16 operand storage saturates
  auto chk = [&](const void* buf, size_t nelems) -> int { return count_saturated(buf, nelems, sat, st); };
  struct StaticWeights {                        // every GEMM below reads prepared weights (see g_tc2_weights_static)
    StaticWeights() { g_tc2_weights_static = true; }
    ~StaticWeights() { g_tc2_weights_static = false; }
  } static_weights_scope;

  {
    cudaStream_t ps = st;
    if (aux) {
      AVSR_CUDA_TRY(cudaEventRecord(aux->fork, st));
      AVSR_CUDA_TRY(cudaStreamWaitEvent(aux->stream, aux->fork, 0));
      ps = aux->stream;
    }
    AVSR_TRY(compute_pos(c, P, W, T, prec, ps));
    if (aux) AVSR_CUDA_TRY(cudaEventRecord(aux->join, ps));
  }
  // v^T pad columns [T, Tp) must be finite (FP32 / TF32 paths; the F16 path keeps V un-transposed)
  if (W.Tp != T && prec != AVSR_PREC_F16)
    AVSR_CUDA_TRY(cudaMemsetAsync(W.vt, 0, (size_t)B * D * W.Tp * sizeof(float), st));

  // FFN w_2 (K = linear_units) as a deferred split-K GEMM: k-slices land in W.splitk and the LayerNorm that follows
  // applies x += 0.5 * (sum of slices + b) while it loads the row.  Not with `taps` (they read x between the two).
  int w2_split = 0;
  const bool w2_defer = prec == AVSR_PREC_F16 && !taps && gemm_tc2_splitk_plan(N, D, F, &w2_split);
  auto w2_parts = [&](const float* bias, float* x_out) {
    LnParts pp;
    pp.part = W.splitk; pp.nparts = w2_split; pp.stride = (long)N * D; pp.bias = bias; pp.alpha = 0.5f; pp.x_out = x_out;
    return pp;
  };

  for (int l = 0; l < L; ++l) {
    const LayerPrep& w = P.layers[l];
    auto tap = [&](int s) -> int {
      if (l == 0 && taps)
        AVSR_CUDA_TRY(cudaMemcpyAsync(taps + (size_t)s * N * D, W.x, stage_bytes, cudaMemcpyDeviceToDevice, st));
      return AVSR_OK;
    };
    // (1) macaron FFN: x += 0.5 * w2(relu(w1 LN(x)))                         conformer_encoder.py:110-116
    // (for l > 0 the norm_ff_macaron output was produced together with the previous layer's norm_final)
    if (l == 0) AVSR_TRY(launch_layernorm(W.x, w.ln_ffm_w, w.ln_ffm_b, W.xn, N, D, opk, st));
    AVSR_TRY(chk(W.xn, (size_t)N * D));
    AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.xn, w.ffm_w1, N, F, D, epi_linear(N, F, w.ffm_b1, W.hid, nullptr, 0.f, 1, opr), st));
    AVSR_TRY(chk(W.hid, (size_t)N * F));
    if (w2_defer) {
      AVSR_TRY(gemm_tc2_splitk(W.hid, w.ffm_w2, N, D, F, W.splitk, w2_split, st));
    } else {
      AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.hid, w.ffm_w2, N, D, F, epi_linear(N, D, w.ffm_b2, W.x, W.x, 0.5f, 0, 0), st));
      AVSR_TRY(tap(0));
    }
    // (2) rel-pos MHA: x += out(attn(LN(x)))                                  conformer_encoder.py:119-142
    {
      const LnParts pp = w2_parts(w.ffm_b2, W.x);
      AVSR_TRY(launch_layernorm(W.x, w.ln_mha_w, w.ln_mha_b, W.xn, N, D, opk, st, w2_defer ? &pp : nullptr));
      AVSR_TRY(chk(W.xn, (size_t)N * D));
    }
    {
      EpiParams e{};
      e.M = N; e.bias = w.qk_b; e.T = T; e.H = H; e.pos_u = w.pos_u; e.pos_v = w.pos_v;
      e.qu = W.qu; e.qv = W.qv; e.kk = W.kk; e.vt = W.vt; e.round_out = opr;
      if (prec == AVSR_PREC_F16) {
        // one QKV projection; V keeps the (B,H,T,64) layout (the P.V MMA reads it as an MN-major operand)
        e.N = 3 * D;
        AVSR_TRY(run_gemm(prec, EPI_QK, W.xn, w.qk_w, N, 3 * D, D, e, st));
      } else {
        e.N = 2 * D;
        AVSR_TRY(run_gemm(prec, EPI_QK, W.xn, w.qk_w, N, 2 * D, D, e, st));
        EpiParams v{};
        v.M = D; v.N = N; v.bias = w.v_b; v.T = T; v.H = H; v.Tp = W.Tp; v.vt = W.vt; v.round_out = opr;
        AVSR_TRY(run_gemm(prec, EPI_VT, op_offset(w.qk_w, (size_t)2 * D * D, prec), W.xn, D, N, D, v, st));
      }
    }
    if (l == 0 && aux) AVSR_CUDA_TRY(cudaStreamWaitEvent(st, aux->join, 0));   // the pos tables are ready
    AVSR_TRY(chk(W.qu, (size_t)N * D)); AVSR_TRY(chk(W.qv, (size_t)N * D));
    AVSR_TRY(chk(W.kk, (size_t)N * D)); AVSR_TRY(chk(W.vt, (size_t)N * D));
    if (l == 0) AVSR_TRY(chk(W.pos, (size_t)L * W.Rp * D / 8 * 8));
    {
      const void* pos_l = op_offset(W.pos, (size_t)l * H * W.Rp * kHeadDim, prec);
      if (prec == AVSR_PREC_F16)
        AVSR_TRY(attention_f16((const __half*)W.qu, (const __half*)W.qv, (const __half*)W.kk, (const __half*)W.vt,
                               (const __half*)pos_l, lengths, (__half*)W.ctx, B, T, H, W.Rp, st));
      else if (prec == AVSR_PREC_TF32)
        AVSR_TRY(attention_tc(W.qu, W.qv, W.kk, W.vt, (const float*)pos_l, lengths, W.ctx, B, T, H, W.Tp, W.Rp, 1, st));
      else
        AVSR_TRY(attention_simt(W.qu, W.qv, W.kk, W.vt, (const float*)pos_l, lengths, W.ctx, B, T, H, W.Tp, W.Rp, 0, st));
    }
    AVSR_TRY(chk(W.ctx, (size_t)N * D));
    AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.ctx, w.out_w, N, D, D, epi_linear(N, D, w.out_b, W.x, W.x, 1.0f, 0, 0), st));
    AVSR_TRY(tap(1));
    // (3) conv module: x += pw2(silu(bn(dw(glu(pw1 LN(x))))))                 conformer_encoder.py:145-151, :30-35
    AVSR_TRY(launch_layernorm(W.x, w.ln_conv_w, w.ln_conv_b, W.xn, N, D, opk, st));
    AVSR_TRY(chk(W.xn, (size_t)N * D));
    {
      EpiParams e{};
      e.M = N; e.N = 2 * D; e.bias = w.pw1_b; e.out = W.glu; e.ldo = D;
      AVSR_TRY(run_gemm(prec, EPI_GLU, W.xn, w.pw1_w, N, 2 * D, D, e, st));
    }
    AVSR_TRY(launch_dwconv_bn_silu(W.glu, w.dw_wt, w.dw_scale, w.dw_shift, W.dw, B, T, D, c.cnn_kernel, opk, st));
    AVSR_TRY(chk(W.dw, (size_t)N * D));
    AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.dw, w.pw2_w, N, D, D, epi_linear(N, D, w.pw2_b, W.x, W.x, 1.0f, 0, 0), st));
    AVSR_TRY(tap(2));
    // (4) FFN: x += 0.5 * w2(relu(w1 LN(x)))                                  conformer_encoder.py:154-159
    AVSR_TRY(launch_layernorm(W.x, w.ln_ff_w, w.ln_ff_b, W.xn, N, D, opk, st));
    AVSR_TRY(chk(W.xn, (size_t)N * D));
    AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.xn, w.ff_w1, N, F, D, epi_linear(N, F, w.ff_b1, W.hid, nullptr, 0.f, 1, opr), st));
    AVSR_TRY(chk(W.hid, (size_t)N * F));
    if (w2_defer) {
      AVSR_TRY(gemm_tc2_splitk(W.hid, w.ff_w2, N, D, F, W.splitk, w2_split, st));
    } else {
      AVSR_TRY(run_gemm(prec, EPI_LINEAR, W.hid, w.ff_w2, N, D, F, epi_linear(N, D, w.ff_b2, W.x, W.x, 0.5f, 0, 0), st));
      AVSR_TRY(tap(3));
    }
    // (5) x = LN_final(x)                                                     conformer_encoder.py:161-162
    //     fused with the next layer's norm_ff_macaron: one pass writes x (fp32) and xn (operand)
    {
      const LnParts pp = w2_parts(w.ff_b2, nullptr);   // the LayerNorm's own fp32 output replaces x
      const LnParts* ppp = w2_defer ? &pp : nullptr;
      if (l + 1 < L) {
        const LayerPrep& nx = P.layers[l + 1];
        AVSR_TRY(launch_layernorm2(W.x, w.ln_fin_w, w.ln_fin_b, nx.ln_ffm_w, nx.ln_ffm_b, W.x, W.xn, N, D, opk, st, ppp));
        // (the next iteration's first check covers this xn)
      } else {
        AVSR_TRY(launch_layernorm(W.x, w.ln_fin_w, w.ln_fin_b, W.x, N, D, OP_F32, st, ppp));
      }
    }
    AVSR_TRY(tap(4));
  }
  return AVSR_OK;
}

static int forward_impl(const AvsrEncoderConfig* cfg, const void* prepared, const float* xs, const int32_t* lengths,
                        int B, int T, float* out, float* taps, void* workspace, size_t workspace_bytes, int precision,
                        void* stream, unsigned long long* sat = nullptr) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  AVSR_REQUIRE(B >= 0 && T >= 0, "bad B=%d T=%d", B, T);
  if (B == 0 || T == 0) return AVSR_OK;  // empty batch: nothing to do
  AVSR_REQUIRE(prepared && xs && out && workspace, "NULL buffer");
  AVSR_REQUIRE((long)B * T < (1L << 24), "B*T=%ld too large", (long)B * T);
  Workspace W = layout_workspace(*cfg, B, T, workspace);
  if (W.bytes > workspace_bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", W.bytes, workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  Prepared P = layout_prepared(*cfg, const_cast<void*>(prepared));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  AVSR_TRY(launch_embed_scale(xs, W.x, (long)B * T * cfg->d_model, sqrtf((float)cfg->d_model), st));
  if (sat) AVSR_CUDA_TRY(cudaMemsetAsync(sat, 0, sizeof(unsigned long long), st));
  AVSR_TRY(forward_body(*cfg, P, W, B, T, lengths, taps, precision, st, nullptr, sat));
  AVSR_TRY(launch_layernorm(W.x, P.after_w, P.after_b, out, B * T, cfg->d_model, 0, st));
  return AVSR_OK;
}

// ------------------------------------------------------------------ the steps either side of the encoder (SURVEY 8f #1)
// proj_encoder = Linear(idim -> d_model) in front (e2e_asr_conformer.py:31,70), ctc_lo = Linear(d_model -> odim) +
// log_softmax behind (ctc.py:21,77-84).  Prepared once per parameter update: proj weights in operand storage, both
// plain and pre-multiplied by sqrt(d_model) (the encoder's embed scale, embedding.py:178, folded into the projection
// that writes the residual stream); ctc_lo weights in operand storage with odim padded to a multiple of 512 (zero
// rows; the pair tile of the two-SM GEMM) and the bias padded likewise.
struct HeadPrep {
  float *proj_w, *proj_b, *proj_ws, *proj_bs, *ctc_w, *ctc_b;
  int npad;
  size_t bytes;
};
static HeadPrep layout_head(const AvsrEncoderConfig& c, int idim, int odim, void* base) {
  HeadPrep H;
  Carver cv{reinterpret_cast<char*>(base)};
  const size_t D = c.d_model;
  H.npad = (int)align_up((size_t)odim, 512);
  H.proj_w = cv.take(D * idim); H.proj_b = cv.take(D);
  H.proj_ws = cv.take(D * idim); H.proj_bs = cv.take(D);
  H.ctc_w = cv.take((size_t)H.npad * D); H.ctc_b = cv.take((size_t)H.npad);
  H.bytes = cv.off;
  return H;
}

struct HeadWorkspace {
  void* enc;          // the encoder's own workspace (layout_workspace)
  size_t enc_bytes;
  float *fx, *logits;
  LsePart* parts;
  size_t bytes;
};
static HeadWorkspace layout_head_workspace(const AvsrEncoderConfig& c, int B, int T, int idim, int odim, void* base) {
  HeadWorkspace W;
  const size_t N = (size_t)B * T;
  const int npad = (int)align_up((size_t)odim, 512);
  W.enc = base;
  W.enc_bytes = align_up(layout_workspace(c, B, T, nullptr).bytes, 256);
  Carver cv{reinterpret_cast<char*>(base) + W.enc_bytes};
  W.fx = cv.take(N * (size_t)(idim > c.d_model ? idim : c.d_model));   // operand copy of the features / of hs
  W.logits = cv.take(N * (size_t)npad);
  W.parts = reinterpret_cast<LsePart*>(cv.take((size_t)2 * (npad / 512) * N * (sizeof(LsePart) / sizeof(float))));
  W.bytes = W.enc_bytes + cv.off;
  return W;
}

// hs_op (rows, d_model) in operand storage -> logp (rows, odim) fp32 log-probabilities [+ arg max]
static int ctc_logprobs(const AvsrEncoderConfig& c, const HeadPrep& H, const void* hs_op, int rows, int odim, float* logits,
                        LsePart* parts, float* logp, int32_t* argmax, int prec, cudaStream_t st) {
  const int D = c.d_model;
  if (prec == AVSR_PREC_F16 && gemm_tc2_lse_ok(rows, H.npad, D)) {
    int nparts = 0;
    AVSR_TRY(gemm_tc2_lse(hs_op, H.ctc_w, H.ctc_b, rows, H.npad, D, odim, logits, H.npad, parts, &nparts, st));
    return launch_lse_finish(logits, H.npad, parts, nparts, rows, logp, odim, argmax, odim, st);
  }
  AVSR_TRY(run_gemm(prec, EPI_LINEAR, hs_op, H.ctc_w, rows, H.npad, D, epi_linear(rows, H.npad, H.ctc_b, logits, nullptr, 0.f, 0, 0), st));
  return launch_log_softmax_rows(logits, H.npad, logp, odim, argmax, rows, odim, st);
}

// features (already resident at `feats`) -> enc_out / logp / argmax: the schedule both the direct call and the captured
// plan run.  `aux` (optional) forks the rel-pos branch like forward_body does.
static int head_forward_body(const AvsrEncoderConfig& c, const Prepared& P, const HeadPrep& H, const Workspace& W,
                             const HeadWorkspace& HW, const float* feats, const int32_t* lengths, int B, int T, int idim,
                             int odim, float* enc_out, float* logp, int32_t* argmax, int precision, cudaStream_t st,
                             const AuxFork* aux) {
  const int N = B * T, D = c.d_model;
  // (1) proj_encoder with the embed scale folded in, straight into the residual stream: x = sqrt(d) * (f Wp^T + bp)
  const void* fx = feats;
  if (precision != AVSR_PREC_FP32) { AVSR_TRY(copy_round(feats, HW.fx, (long)N * idim, operand_kind(precision), st)); fx = HW.fx; }
  AVSR_TRY(run_gemm(precision, EPI_LINEAR, fx, H.proj_ws, N, D, idim, epi_linear(N, D, H.proj_bs, W.x, nullptr, 0.f, 0, 0), st));
  // (2) the 12 layers
  AVSR_TRY(forward_body(c, P, W, B, T, lengths, nullptr, precision, st, aux));
  // (3) after_norm: fp32 features for the caller (attention decoder / beam search) + the operand of ctc_lo in one pass
  float* feat_out = enc_out ? enc_out : W.x;
  AVSR_TRY(launch_layernorm_dual(W.x, P.after_w, P.after_b, feat_out, W.xn, N, D, operand_kind(precision), st));
  // (4) ctc_lo + log_softmax: GEMM with log-sum-exp partials in its epilogue, one finishing pass
  return ctc_logprobs(c, H, W.xn, N, odim, HW.logits, HW.parts, logp, argmax, precision, st);
}

}  // namespace avsr

// ====================================================================== C ABI
using namespace avsr;

struct AvsrPlan {
  AvsrEncoderConfig cfg;
  Prepared P;
  Workspace W;
  int B, T, precision;
  float* head_feats = nullptr;     // head plans: staging copy of the features inside the plan's workspace
  int head_idim = 0;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  uint64_t kernel_nodes = 0;       // launches one replay adds to avsr_launch_count
};

static uint64_t graph_kernel_nodes(cudaGraph_t g) {
  size_t n = 0;
  if (cudaGraphGetNodes(g, nullptr, &n) != cudaSuccess) return 0;
  std::vector<cudaGraphNode_t> nodes(n);
  if (n == 0 || cudaGraphGetNodes(g, nodes.data(), &n) != cudaSuccess) return 0;
  uint64_t k = 0;
  for (auto nd : nodes) {
    cudaGraphNodeType t;
    if (cudaGraphNodeGetType(nd, &t) == cudaSuccess && t == cudaGraphNodeTypeKernel) ++k;
  }
  return k;
}

// Records `body(aux)` -- the schedule on `st`, with the rel-pos branch forked onto `aux` -- into p->graph / p->exec.
// The body runs once outside capture first (function attributes such as the dynamic shared-memory opt-in must not be
// set lazily during capture; lazy module loading), then is captured; the captured launches are counted when the graph
// is replayed.  The auxiliary stream and events live for the duration of the call.  On error nothing is left behind
// but `p` itself, which the caller deletes.
template <typename Body>
static int capture_plan(AvsrPlan* p, cudaStream_t st, Body&& body) {
  AuxFork aux;
  int rc = AVSR_OK;
  if (cudaStreamCreateWithFlags(&aux.stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&aux.fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&aux.join, cudaEventDisableTiming) != cudaSuccess) {
    set_error("plan: cannot create the auxiliary stream / events: %s", cudaGetErrorString(cudaGetLastError()));
    rc = AVSR_E_CUDA;
  }
  if (rc == AVSR_OK) rc = body(&aux);
  if (rc == AVSR_OK && (cudaStreamSynchronize(st) != cudaSuccess || cudaStreamSynchronize(aux.stream) != cudaSuccess)) {
    set_error("plan warm-up failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = AVSR_E_CUDA;
  }
  if (rc == AVSR_OK) {
    cudaError_t e = cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) {
      set_error("cudaStreamBeginCapture: %s", cudaGetErrorString(e));
      rc = AVSR_E_CUDA;
    } else {
      const uint64_t before = g_launches.load();
      rc = body(&aux);   // the aux stream joins the capture through the fork event
      g_launches.store(before);
      e = cudaStreamEndCapture(st, &p->graph);
      if (rc == AVSR_OK && e != cudaSuccess) { set_error("cudaStreamEndCapture: %s", cudaGetErrorString(e)); rc = AVSR_E_CUDA; }
    }
  }
  if (rc == AVSR_OK) {
    const cudaError_t e = cudaGraphInstantiate(&p->exec, p->graph, 0);
    if (e != cudaSuccess) { set_error("cudaGraphInstantiate: %s", cudaGetErrorString(e)); rc = AVSR_E_CUDA; }
  }
  if (aux.join) cudaEventDestroy(aux.join);
  if (aux.fork) cudaEventDestroy(aux.fork);
  if (aux.stream) cudaStreamDestroy(aux.stream);
  if (rc != AVSR_OK) {
    if (p->graph) cudaGraphDestroy(p->graph);
    p->graph = nullptr;
    return rc;
  }
  p->kernel_nodes = graph_kernel_nodes(p->graph);
  return AVSR_OK;
}

#ifdef AVSR_TRACE
namespace avsr {
int trace_bind_gemm_tc2(unsigned long long*);
int trace_bind_attention_f16(unsigned long long*);
int trace_bind_elementwise(unsigned long long*);
int trace_bind_gemm_tc(unsigned long long*);
static int trace_bind_all(unsigned long long* p) {
  return trace_bind_gemm_tc2(p) | trace_bind_attention_f16(p) | trace_bind_elementwise(p) | trace_bind_gemm_tc(p);
}
}
// diagnostic build only (scripts/build_trace.py): device buffer of `words` 64-bit words, see common.cuh "phase trace"
extern "C" int avsr_trace_set(void* device_buffer, size_t words, void* stream) {
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!device_buffer || words < 2 + (size_t)kTraceWords) {
    AVSR_CUDA_TRY(cudaDeviceSynchronize());
    AVSR_REQUIRE(avsr::trace_bind_all(nullptr) == 0, "trace: cannot unbind");
    return AVSR_OK;
  }
  const unsigned long long head[2] = {0ULL, (unsigned long long)((words - 2) / kTraceWords)};
  AVSR_CUDA_TRY(cudaMemsetAsync(device_buffer, 0, words * 8, st));
  AVSR_CUDA_TRY(cudaMemcpyAsync(device_buffer, head, sizeof(head), cudaMemcpyHostToDevice, st));
  AVSR_CUDA_TRY(cudaStreamSynchronize(st));
  AVSR_REQUIRE(avsr::trace_bind_all(reinterpret_cast<unsigned long long*>(device_buffer)) == 0, "trace: cannot bind");
  return AVSR_OK;
}
#endif

extern "C" {

int avsr_abi_version(void) { return AVSR_ABI_VERSION; }
const char* avsr_last_error(void) { return g_err.c_str(); }
uint64_t avsr_launch_count(void) { return g_launches.load(); }

size_t avsr_prepared_bytes(const AvsrEncoderConfig* cfg) {
  if (check_cfg(cfg) != AVSR_OK) return 0;
  return layout_prepared(*cfg, nullptr).bytes;
}

int avsr_prepare_weights(const AvsrEncoderConfig* cfg, const AvsrLayerParams* layers, const float* after_norm_w,
                         const float* after_norm_b, void* prepared, size_t prepared_bytes, int precision,
                         void* stream) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(layers && after_norm_w && after_norm_b && prepared, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  Prepared P = layout_prepared(*cfg, prepared);
  if (P.bytes > prepared_bytes) {
    set_error("prepared buffer too small: need %zu bytes, got %zu", P.bytes, prepared_bytes);
    return AVSR_E_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int rnd = operand_kind(precision);   // storage kind of the GEMM weights
  const long D = cfg->d_model, F = cfg->linear_units, K = cfg->cnn_kernel;
  for (int l = 0; l < cfg->num_blocks; ++l) {
    const AvsrLayerParams& s = layers[l];
    const LayerPrep& d = P.layers[l];
    const float* const* sp = reinterpret_cast<const float* const*>(&s);
    for (size_t i = 0; i < sizeof(AvsrLayerParams) / sizeof(float*); ++i)
      AVSR_REQUIRE(sp[i] != nullptr, "layer %d: parameter pointer #%zu is NULL", l, i);
    AVSR_TRY(copy_round(s.ffm_w1, d.ffm_w1, F * D, rnd, st)); AVSR_TRY(copy_round(s.ffm_b1, d.ffm_b1, F, 0, st));
    AVSR_TRY(copy_round(s.ffm_w2, d.ffm_w2, D * F, rnd, st)); AVSR_TRY(copy_round(s.ffm_b2, d.ffm_b2, D, 0, st));
    AVSR_TRY(copy_round(s.norm_ffm_w, d.ln_ffm_w, D, 0, st)); AVSR_TRY(copy_round(s.norm_ffm_b, d.ln_ffm_b, D, 0, st));
    AVSR_TRY(copy_round(s.q_w, d.qk_w, D * D, rnd, st)); AVSR_TRY(copy_round(s.k_w, op_offset(d.qk_w, (size_t)D * D, precision), D * D, rnd, st));
    AVSR_TRY(copy_round(s.q_b, d.qk_b, D, 0, st)); AVSR_TRY(copy_round(s.k_b, d.qk_b + D, D, 0, st));
    AVSR_TRY(copy_round(s.v_w, op_offset(d.qk_w, (size_t)2 * D * D, precision), D * D, rnd, st));
    AVSR_TRY(copy_round(s.v_b, d.qk_b + 2 * D, D, 0, st));
    AVSR_TRY(copy_round(s.out_w, d.out_w, D * D, rnd, st)); AVSR_TRY(copy_round(s.out_b, d.out_b, D, 0, st));
    AVSR_TRY(copy_round(s.pos_bias_u, d.pos_u, D, 0, st)); AVSR_TRY(copy_round(s.pos_bias_v, d.pos_v, D, 0, st));
    AVSR_TRY(copy_round(s.norm_mha_w, d.ln_mha_w, D, 0, st)); AVSR_TRY(copy_round(s.norm_mha_b, d.ln_mha_b, D, 0, st));
    glu_interleave_kernel<<<(unsigned)(2 * D), 256, 0, st>>>(s.pw1_w, s.pw1_b, d.pw1_w, d.pw1_b, (int)D, rnd);
    AVSR_CHECK_LAUNCH();
    dw_fold_kernel<<<cdiv((int)D, 128), 128, 0, st>>>(s.dw_w, s.dw_b, s.bn_w, s.bn_b, s.bn_mean, s.bn_var, d.dw_wt,
                                                      d.dw_scale, d.dw_shift, (int)D, (int)K);
    AVSR_CHECK_LAUNCH();
    AVSR_TRY(copy_round(s.pw2_w, d.pw2_w, D * D, rnd, st)); AVSR_TRY(copy_round(s.pw2_b, d.pw2_b, D, 0, st));
    AVSR_TRY(copy_round(s.norm_conv_w, d.ln_conv_w, D, 0, st)); AVSR_TRY(copy_round(s.norm_conv_b, d.ln_conv_b, D, 0, st));
    AVSR_TRY(copy_round(s.ff_w1, d.ff_w1, F * D, rnd, st)); AVSR_TRY(copy_round(s.ff_b1, d.ff_b1, F, 0, st));
    AVSR_TRY(copy_round(s.ff_w2, d.ff_w2, D * F, rnd, st)); AVSR_TRY(copy_round(s.ff_b2, d.ff_b2, D, 0, st));
    AVSR_TRY(copy_round(s.norm_ff_w, d.ln_ff_w, D, 0, st)); AVSR_TRY(copy_round(s.norm_ff_b, d.ln_ff_b, D, 0, st));
    AVSR_TRY(copy_round(s.norm_final_w, d.ln_fin_w, D, 0, st)); AVSR_TRY(copy_round(s.norm_final_b, d.ln_fin_b, D, 0, st));
    AVSR_TRY(copy_round(s.pos_w, op_offset(P.pos_w_all, (size_t)l * D * D, precision), D * D, rnd, st));
  }
  AVSR_TRY(copy_round(after_norm_w, P.after_w, D, 0, st));
  AVSR_TRY(copy_round(after_norm_b, P.after_b, D, 0, st));
  return AVSR_OK;
}

size_t avsr_workspace_bytes(const AvsrEncoderConfig* cfg, int B, int T) {
  if (check_cfg(cfg) != AVSR_OK || B < 0 || T < 0) return 0;
  if (B == 0 || T == 0) return 256;
  return layout_workspace(*cfg, B, T, nullptr).bytes;
}

int avsr_encoder_forward(const AvsrEncoderConfig* cfg, const void* prepared, const float* xs, const int32_t* lengths,
                         int B, int T, float* out, void* workspace, size_t workspace_bytes, int precision,
                         void* stream) {
  return forward_impl(cfg, prepared, xs, lengths, B, T, out, nullptr, workspace, workspace_bytes, precision, stream);
}

int avsr_encoder_forward_checked(const AvsrEncoderConfig* cfg, const void* prepared, const float* xs,
                                 const int32_t* lengths, int B, int T, float* out, void* workspace,
                                 size_t workspace_bytes, int precision, uint64_t* saturated, void* stream) {
  AVSR_REQUIRE(saturated != nullptr, "saturated counter is NULL");
  return forward_impl(cfg, prepared, xs, lengths, B, T, out, nullptr, workspace, workspace_bytes, precision, stream,
                      reinterpret_cast<unsigned long long*>(saturated));
}

int avsr_encoder_forward_taps(const AvsrEncoderConfig* cfg, const void* prepared, const float* xs,
                              const int32_t* lengths, int B, int T, float* out, float* taps, void* workspace,
                              size_t workspace_bytes, int precision, void* stream) {
  return forward_impl(cfg, prepared, xs, lengths, B, T, out, taps, workspace, workspace_bytes, precision, stream);
}

int avsr_plan_create(const AvsrEncoderConfig* cfg, const void* prepared, int B, int T, void* workspace,
                     size_t workspace_bytes, int precision, void* stream, AvsrPlan** plan) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(plan && prepared && workspace, "NULL argument");
  AVSR_REQUIRE(B > 0 && T > 0, "plan needs B>0, T>0 (got %d, %d)", B, T);
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  Workspace W = layout_workspace(*cfg, B, T, workspace);
  if (W.bytes > workspace_bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", W.bytes, workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  AvsrPlan* p = new AvsrPlan();
  p->cfg = *cfg; p->B = B; p->T = T; p->precision = precision; p->W = W;
  p->P = layout_prepared(*cfg, const_cast<void*>(prepared));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  fill_lengths_kernel<<<cdiv(B, 128), 128, 0, st>>>(W.lengths, nullptr, B, T);
  g_launches.fetch_add(1);
  const int rc = capture_plan(p, st, [&](const AuxFork* aux) {
    return forward_body(p->cfg, p->P, p->W, B, T, p->W.lengths, nullptr, precision, st, aux);
  });
  if (rc != AVSR_OK) { delete p; return rc; }
  *plan = p;
  return AVSR_OK;
}

int avsr_plan_forward(AvsrPlan* p, const float* xs, const int32_t* lengths, float* out, void* stream) {
  AVSR_REQUIRE(p && xs && out, "NULL argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int N = p->B * p->T, D = p->cfg.d_model;
  fill_lengths_kernel<<<cdiv(p->B, 128), 128, 0, st>>>(p->W.lengths, lengths, p->B, p->T);
  AVSR_CHECK_LAUNCH();
  AVSR_TRY(launch_embed_scale(xs, p->W.x, (long)N * D, sqrtf((float)D), st));
  AVSR_CUDA_TRY(cudaGraphLaunch(p->exec, st));
  g_launches.fetch_add(p->kernel_nodes);
  AVSR_TRY(launch_layernorm(p->W.x, p->P.after_w, p->P.after_b, out, N, D, 0, st));
  return AVSR_OK;
}

void avsr_plan_destroy(AvsrPlan* p) {
  if (!p) return;
  if (p->exec) cudaGraphExecDestroy(p->exec);
  if (p->graph) cudaGraphDestroy(p->graph);
  delete p;
}

// ---------------------------------------------------------------------- per-op entry points
int avsr_layernorm(const float* x, const float* gamma, const float* beta, float* y, int rows, int d, void* stream) {
  AVSR_REQUIRE(x && gamma && beta && y, "NULL argument");
  return launch_layernorm(x, gamma, beta, y, rows, d, 0, reinterpret_cast<cudaStream_t>(stream));
}

size_t avsr_linear_workspace_bytes(int rows, int n, int k, int precision) {
  if (precision != AVSR_PREC_F16 || rows <= 0 || n <= 0 || k <= 0) return 16;
  return align_up((size_t)rows * k * 2, 256) + align_up((size_t)n * k * 2, 256);
}

int avsr_linear(const float* x, const float* w, const float* bias, const float* resid, float alpha, int relu, float* y,
                int rows, int n, int k, int precision, void* workspace, size_t workspace_bytes, void* stream) {
  AVSR_REQUIRE(x && w && y, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const void *xa = x, *wa = w;
  if (precision == AVSR_PREC_F16 && rows > 0 && n > 0) {
    AVSR_REQUIRE(workspace != nullptr, "avsr_linear: AVSR_PREC_F16 needs a workspace");
    if (avsr_linear_workspace_bytes(rows, n, k, precision) > workspace_bytes) {
      set_error("linear workspace too small: need %zu bytes, got %zu", avsr_linear_workspace_bytes(rows, n, k, precision),
                workspace_bytes);
      return AVSR_E_WORKSPACE;
    }
    char* xh = reinterpret_cast<char*>(workspace);
    char* wh = xh + align_up((size_t)rows * k * 2, 256);
    AVSR_TRY(copy_round(x, xh, (long)rows * k, OP_F16, st));
    AVSR_TRY(copy_round(w, wh, (long)n * k, OP_F16, st));
    xa = xh; wa = wh;
  }
  // note: in TF32 mode operands are used as given (the tensor core truncates fp32 -> tf32)
  return run_gemm(precision, EPI_LINEAR, xa, wa, rows, n, k, epi_linear(rows, n, bias, y, resid, alpha, relu, 0), st);
}

int avsr_linear_operands(const void* x_op, const void* w_op, const float* bias, const float* resid, float alpha,
                         void* y, int rows, int n, int k, int relu, int y_is_operand, int precision, void* stream) {
  AVSR_REQUIRE(x_op && w_op && y, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  return run_gemm(precision, EPI_LINEAR, x_op, w_op, rows, n, k,
                  epi_linear(rows, n, bias, y, resid, alpha, relu, (y_is_operand && precision != AVSR_PREC_FP32) ? 1 : 0),
                  reinterpret_cast<cudaStream_t>(stream));
}

// (B,T,H*64) -> (B,H,T,64) with optional per-channel bias add; or -> (B,H,64,Tp) when transpose != 0
__global__ void split_heads_kernel(const float* __restrict__ src, const float* __restrict__ bias, void* __restrict__ dst,
                                   int B, int T, int H, int Tp, int transpose, int kind) {
  const long total = (long)B * T * H * kHeadDim;
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int c = (int)(i % (H * kHeadDim));
    const long r = i / (H * kHeadDim);
    const int b = (int)(r / T), t = (int)(r % T), h = c / kHeadDim, d = c % kHeadDim;
    const float v = src[i] + (bias ? bias[c] : 0.f);
    const long o = transpose ? (((long)b * H + h) * kHeadDim + d) * Tp + t : (((long)b * H + h) * T + t) * kHeadDim + d;
    if (kind == OP_F16) reinterpret_cast<__half*>(dst)[o] = to_half_sat(v);
    else reinterpret_cast<float*>(dst)[o] = kind == OP_TF32 ? round_tf32(v) : v;
  }
}

__global__ void half_to_float_kernel(const __half* __restrict__ src, float* __restrict__ dst, long n) {
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    dst[i] = __half2float(src[i]);
}

size_t avsr_attention_workspace_bytes(int B, int T, int H) {
  if (B <= 0 || T <= 0 || H <= 0) return 256;
  const size_t N = (size_t)B * T, D = (size_t)H * kHeadDim, Tp = (T + 7) & ~7;
  return 4 * align_up(N * D * 4, 256) + align_up((size_t)B * D * Tp * 4, 256) + align_up((size_t)(2 * T - 1) * D * 4, 256);
}

int avsr_relpos_attention(const float* q, const float* k, const float* v, const float* p, const float* pos_bias_u,
                          const float* pos_bias_v, const int32_t* lengths, float* ctx, int B, int T, int H,
                          void* workspace, size_t workspace_bytes, int precision, void* stream) {
  AVSR_REQUIRE(q && k && v && p && pos_bias_u && pos_bias_v && ctx && workspace, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  if (B <= 0 || T <= 0) return AVSR_OK;
  if (avsr_attention_workspace_bytes(B, T, H) > workspace_bytes) {
    set_error("attention workspace too small: need %zu, got %zu", avsr_attention_workspace_bytes(B, T, H), workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const size_t N = (size_t)B * T, D = (size_t)H * kHeadDim;
  const int Tp = (T + 7) & ~7, R = 2 * T - 1;
  const int kind = operand_kind(precision);
  Carver cv{reinterpret_cast<char*>(workspace)};
  float *qu = cv.take(N * D), *qv = cv.take(N * D), *kk = cv.take(N * D), *vt = cv.take((size_t)B * D * Tp),
        *pos = cv.take((size_t)R * D), *ctxh = cv.take(N * D);
  const int blocks = 148 * 4;
  if (Tp != T) AVSR_CUDA_TRY(cudaMemsetAsync(vt, 0, (size_t)B * D * Tp * sizeof(float), st));
  split_heads_kernel<<<blocks, 256, 0, st>>>(q, pos_bias_u, qu, B, T, H, Tp, 0, kind); AVSR_CHECK_LAUNCH();
  split_heads_kernel<<<blocks, 256, 0, st>>>(q, pos_bias_v, qv, B, T, H, Tp, 0, kind); AVSR_CHECK_LAUNCH();
  split_heads_kernel<<<blocks, 256, 0, st>>>(k, nullptr, kk, B, T, H, Tp, 0, kind); AVSR_CHECK_LAUNCH();
  split_heads_kernel<<<blocks, 256, 0, st>>>(v, nullptr, vt, B, T, H, Tp, precision == AVSR_PREC_F16 ? 0 : 1, kind);
  AVSR_CHECK_LAUNCH();
  split_heads_kernel<<<blocks, 256, 0, st>>>(p, nullptr, pos, 1, R, H, R, 0, kind); AVSR_CHECK_LAUNCH();
  if (precision == AVSR_PREC_F16) {
    AVSR_TRY(attention_f16((const __half*)qu, (const __half*)qv, (const __half*)kk, (const __half*)vt, (const __half*)pos,
                           lengths, (__half*)ctxh, B, T, H, R, st));
    half_to_float_kernel<<<blocks, 256, 0, st>>>((const __half*)ctxh, ctx, (long)N * D);
    AVSR_CHECK_LAUNCH();
    return AVSR_OK;
  }
  if (precision == AVSR_PREC_TF32) return attention_tc(qu, qv, kk, vt, pos, lengths, ctx, B, T, H, Tp, R, 0, st);
  return attention_simt(qu, qv, kk, vt, pos, lengths, ctx, B, T, H, Tp, R, 0, st);
}

int avsr_dwconv_bn_silu(const float* x, const float* w, const float* b, const float* bn_w, const float* bn_b,
                        const float* bn_mean, const float* bn_var, float* y, int B, int T, int C, int K,
                        void* workspace, size_t workspace_bytes, void* stream) {
  AVSR_REQUIRE(x && w && b && bn_w && bn_b && bn_mean && bn_var && y && workspace, "NULL argument");
  AVSR_REQUIRE(C > 0 && C % 4 == 0 && K >= 1 && K % 2 == 1, "dwconv: bad C=%d K=%d", C, K);
  if ((size_t)(K + 2) * C * sizeof(float) > workspace_bytes) {
    set_error("dwconv workspace too small: need %zu bytes, got %zu", (size_t)(K + 2) * C * sizeof(float), workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float *wt = reinterpret_cast<float*>(workspace), *scale = wt + (size_t)K * C, *shift = scale + C;
  dw_fold_kernel<<<cdiv(C, 128), 128, 0, st>>>(w, b, bn_w, bn_b, bn_mean, bn_var, wt, scale, shift, C, K);
  AVSR_CHECK_LAUNCH();
  return launch_dwconv_bn_silu(x, wt, scale, shift, y, B, T, C, K, 0, st);
}

size_t avsr_pointwise_glu_workspace_bytes(int rows, int C) {
  if (rows < 0 || C <= 0) return 16;
  return align_up(((size_t)2 * C * C + 2 * C) * sizeof(float), 256) + align_up((size_t)rows * C * 2, 256);
}

int avsr_pointwise_glu(const float* x, const float* w, const float* b, float* y, int rows, int C, void* workspace,
                       size_t workspace_bytes, int precision, void* stream) {
  AVSR_REQUIRE(x && w && b && y && workspace, "NULL argument");
  AVSR_REQUIRE(C > 0 && C % 64 == 0, "pointwise_glu: C=%d must be a multiple of 64", C);
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  if (avsr_pointwise_glu_workspace_bytes(rows, C) > workspace_bytes) {
    set_error("pointwise_glu workspace too small: need %zu bytes, got %zu", avsr_pointwise_glu_workspace_bytes(rows, C),
              workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  float* wi = reinterpret_cast<float*>(workspace);
  float* bi = wi + (size_t)2 * C * C;
  char* xh = reinterpret_cast<char*>(workspace) + align_up(((size_t)2 * C * C + 2 * C) * sizeof(float), 256);
  const int kind = precision == AVSR_PREC_F16 ? OP_F16 : OP_F32;   // TF32: the tensor core truncates raw fp32
  glu_interleave_kernel<<<(unsigned)(2 * C), 256, 0, st>>>(w, b, wi, bi, C, kind);
  AVSR_CHECK_LAUNCH();
  const void* xa = x;
  if (precision == AVSR_PREC_F16 && rows > 0) {
    AVSR_TRY(copy_round(x, xh, (long)rows * C, OP_F16, st));
    xa = xh;
  }
  EpiParams e{};
  e.M = rows; e.N = 2 * C; e.bias = bi; e.out = y; e.ldo = C;
  return run_gemm(precision, EPI_GLU, xa, wi, rows, 2 * C, C, e, st);
}

size_t avsr_head_prepared_bytes(const AvsrEncoderConfig* cfg, int idim, int odim) {
  if (check_cfg(cfg) != AVSR_OK || idim <= 0 || odim <= 0) return 0;
  return layout_head(*cfg, idim, odim, nullptr).bytes;
}

int avsr_prepare_head(const AvsrEncoderConfig* cfg, int idim, int odim, const float* proj_w, const float* proj_b,
                      const float* ctc_w, const float* ctc_b, void* prepared_head, size_t prepared_bytes, int precision,
                      void* stream) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(prepared_head && ((proj_w && proj_b) || (ctc_w && ctc_b)), "NULL argument");
  AVSR_REQUIRE((!proj_w) == (!proj_b) && (!ctc_w) == (!ctc_b), "weight / bias of a projection must be given together");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  AVSR_REQUIRE(idim > 0 && idim % 8 == 0 && odim > 0, "head: idim=%d must be a positive multiple of 8, odim=%d > 0", idim, odim);
  HeadPrep H = layout_head(*cfg, idim, odim, prepared_head);
  if (H.bytes > prepared_bytes) {
    set_error("prepared head buffer too small: need %zu bytes, got %zu", H.bytes, prepared_bytes);
    return AVSR_E_WORKSPACE;
  }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int rnd = operand_kind(precision);
  const long D = cfg->d_model;
  const float sc = sqrtf((float)cfg->d_model);
  AVSR_CUDA_TRY(cudaMemsetAsync(prepared_head, 0, H.bytes, st));      // zero rows / bias entries of the odim padding
  if (proj_w) {   // a module that owns only one of the two projections prepares its half (the other stays zero)
    AVSR_TRY(copy_round(proj_w, H.proj_w, D * idim, rnd, st)); AVSR_TRY(copy_round(proj_b, H.proj_b, D, 0, st));
    AVSR_TRY(copy_round(proj_w, H.proj_ws, D * idim, rnd, st, sc)); AVSR_TRY(copy_round(proj_b, H.proj_bs, D, 0, st, sc));
  }
  if (ctc_w) {
    AVSR_TRY(copy_round(ctc_w, H.ctc_w, (long)odim * D, rnd, st)); AVSR_TRY(copy_round(ctc_b, H.ctc_b, odim, 0, st));
  }
  return AVSR_OK;
}

size_t avsr_head_workspace_bytes(const AvsrEncoderConfig* cfg, int B, int T, int idim, int odim) {
  if (check_cfg(cfg) != AVSR_OK || B < 0 || T < 0 || idim <= 0 || odim <= 0) return 0;
  if (B == 0 || T == 0) return 256;
  return layout_head_workspace(*cfg, B, T, idim, odim, nullptr).bytes;
}

int avsr_proj_encoder(const AvsrEncoderConfig* cfg, const void* prepared_head, const float* feats, int rows, int idim,
                      int odim, float* y, void* workspace, size_t workspace_bytes, int precision, void* stream) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(prepared_head && feats && y && workspace, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  if (rows <= 0) return AVSR_OK;
  HeadPrep H = layout_head(*cfg, idim, odim, const_cast<void*>(prepared_head));
  const size_t need = align_up((size_t)rows * idim * sizeof(float), 256);
  if (need > workspace_bytes) { set_error("proj_encoder workspace too small: need %zu, got %zu", need, workspace_bytes); return AVSR_E_WORKSPACE; }
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const void* fx = feats;
  if (precision != AVSR_PREC_FP32) { AVSR_TRY(copy_round(feats, workspace, (long)rows * idim, operand_kind(precision), st)); fx = workspace; }
  return run_gemm(precision, EPI_LINEAR, fx, H.proj_w, rows, cfg->d_model, idim,
                  epi_linear(rows, cfg->d_model, H.proj_b, y, nullptr, 0.f, 0, 0), st);
}

size_t avsr_ctc_workspace_bytes(const AvsrEncoderConfig* cfg, int rows, int odim) {
  if (check_cfg(cfg) != AVSR_OK || rows < 0 || odim <= 0) return 0;
  const size_t npad = align_up((size_t)odim, 512);
  return align_up((size_t)rows * cfg->d_model * 4, 256) + align_up((size_t)rows * npad * 4, 256) +
         align_up((size_t)2 * (npad / 512) * rows * sizeof(LsePart), 256) + 256;
}

int avsr_ctc_logprobs(const AvsrEncoderConfig* cfg, const void* prepared_head, const float* hs, int rows, int idim,
                      int odim, float* logp, int32_t* argmax, void* workspace, size_t workspace_bytes, int precision,
                      void* stream) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(prepared_head && hs && (logp || argmax) && workspace, "NULL argument");
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  if (rows <= 0) return AVSR_OK;
  if (avsr_ctc_workspace_bytes(cfg, rows, odim) > workspace_bytes) {
    set_error("ctc workspace too small: need %zu, got %zu", avsr_ctc_workspace_bytes(cfg, rows, odim), workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  HeadPrep H = layout_head(*cfg, idim, odim, const_cast<void*>(prepared_head));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  Carver cv{reinterpret_cast<char*>(workspace)};
  float* hx = cv.take((size_t)rows * cfg->d_model);
  float* logits = cv.take((size_t)rows * H.npad);
  LsePart* parts = reinterpret_cast<LsePart*>(cv.take((size_t)2 * (H.npad / 512) * rows * (sizeof(LsePart) / sizeof(float))));
  const void* hs_op = hs;
  if (precision != AVSR_PREC_FP32) { AVSR_TRY(copy_round(hs, hx, (long)rows * cfg->d_model, operand_kind(precision), st)); hs_op = hx; }
  return ctc_logprobs(*cfg, H, hs_op, rows, odim, logits, parts, logp, argmax, precision, st);
}

int avsr_features_to_logprobs(const AvsrEncoderConfig* cfg, const void* prepared, const void* prepared_head,
                              const float* feats, const int32_t* lengths, int B, int T, int idim, int odim,
                              float* enc_out, float* logp, int32_t* argmax, void* workspace, size_t workspace_bytes,
                              int precision, void* stream) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  AVSR_REQUIRE(B >= 0 && T >= 0 && idim > 0 && odim > 0, "bad B=%d T=%d idim=%d odim=%d", B, T, idim, odim);
  if (B == 0 || T == 0) return AVSR_OK;
  AVSR_REQUIRE(prepared && prepared_head && feats && (logp || argmax) && workspace, "NULL buffer");
  AVSR_REQUIRE((long)B * T < (1L << 24), "B*T=%ld too large", (long)B * T);
  HeadWorkspace HW = layout_head_workspace(*cfg, B, T, idim, odim, workspace);
  if (HW.bytes > workspace_bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", HW.bytes, workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  Workspace W = layout_workspace(*cfg, B, T, HW.enc);
  Prepared P = layout_prepared(*cfg, const_cast<void*>(prepared));
  HeadPrep H = layout_head(*cfg, idim, odim, const_cast<void*>(prepared_head));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  return head_forward_body(*cfg, P, H, W, HW, feats, lengths, B, T, idim, odim, enc_out, logp, argmax, precision, st, nullptr);
}

// The same call replayed from a CUDA graph.  The plan bakes in its buffers: `workspace` (>= avsr_head_plan_workspace_bytes:
// the head workspace + a staging copy of the features + the lengths) and the OUTPUT buffers enc_out / logp / argmax given
// here -- every avsr_head_plan_forward writes into those same buffers.
size_t avsr_head_plan_workspace_bytes(const AvsrEncoderConfig* cfg, int B, int T, int idim, int odim) {
  if (check_cfg(cfg) != AVSR_OK || B <= 0 || T <= 0 || idim <= 0 || odim <= 0) return 0;
  return layout_head_workspace(*cfg, B, T, idim, odim, nullptr).bytes + align_up((size_t)B * T * idim * sizeof(float), 256) + 256;
}

int avsr_head_plan_create(const AvsrEncoderConfig* cfg, const void* prepared, const void* prepared_head, int B, int T,
                          int idim, int odim, float* enc_out, float* logp, int32_t* argmax, void* workspace,
                          size_t workspace_bytes, int precision, void* stream, AvsrPlan** plan) {
  AVSR_TRY(check_cfg(cfg));
  AVSR_REQUIRE(plan && prepared && prepared_head && workspace && (logp || argmax), "NULL argument");
  AVSR_REQUIRE(B > 0 && T > 0 && idim > 0 && odim > 0, "plan needs B>0, T>0 (got %d, %d)", B, T);
  AVSR_REQUIRE(valid_precision(precision), "bad precision %d", precision);
  if (avsr_head_plan_workspace_bytes(cfg, B, T, idim, odim) > workspace_bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", avsr_head_plan_workspace_bytes(cfg, B, T, idim, odim), workspace_bytes);
    return AVSR_E_WORKSPACE;
  }
  HeadWorkspace HW = layout_head_workspace(*cfg, B, T, idim, odim, workspace);
  float* feats_static = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + align_up(HW.bytes, 256));
  AvsrPlan* p = new AvsrPlan();
  p->cfg = *cfg; p->B = B; p->T = T; p->precision = precision;
  p->W = layout_workspace(*cfg, B, T, HW.enc);
  p->P = layout_prepared(*cfg, const_cast<void*>(prepared));
  p->head_feats = feats_static; p->head_idim = idim;
  const HeadPrep H = layout_head(*cfg, idim, odim, const_cast<void*>(prepared_head));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  fill_lengths_kernel<<<cdiv(B, 128), 128, 0, st>>>(p->W.lengths, nullptr, B, T);
  g_launches.fetch_add(1);
  AVSR_CUDA_TRY(cudaMemsetAsync(feats_static, 0, (size_t)B * T * idim * sizeof(float), st));
  const int rc = capture_plan(p, st, [&](const AuxFork* aux) {
    return head_forward_body(p->cfg, p->P, H, p->W, HW, feats_static, p->W.lengths, B, T, idim, odim, enc_out, logp, argmax,
                             precision, st, aux);
  });
  if (rc != AVSR_OK) { delete p; return rc; }
  *plan = p;
  return AVSR_OK;
}

int avsr_head_plan_forward(AvsrPlan* p, const float* feats, const int32_t* lengths, void* stream) {
  AVSR_REQUIRE(p && feats && p->head_feats, "NULL argument / not a head plan");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  fill_lengths_kernel<<<cdiv(p->B, 128), 128, 0, st>>>(p->W.lengths, lengths, p->B, p->T);
  AVSR_CHECK_LAUNCH();
  AVSR_CUDA_TRY(cudaMemcpyAsync(p->head_feats, feats, (size_t)p->B * p->T * p->head_idim * sizeof(float), cudaMemcpyDeviceToDevice, st));
  AVSR_CUDA_TRY(cudaGraphLaunch(p->exec, st));
  g_launches.fetch_add(p->kernel_nodes);
  return AVSR_OK;
}

int avsr_rel_sinusoid_table(float* pe, int T, int d, void* stream) {
  AVSR_REQUIRE(pe, "NULL argument");
  return launch_sinusoid(pe, T, d, 0, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"
