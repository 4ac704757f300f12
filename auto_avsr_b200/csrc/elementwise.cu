// HBM-bound kernels of the Conformer layer: embed scale, LayerNorm, rel-pos sinusoid table,
// depthwise-conv + BatchNorm(eval) + SiLU.  fp32 math; coalesced float4 accesses along the channel axis
// (channels are the contiguous axis of the reference's (B,T,C) layout, so a warp reads 512 contiguous bytes).
#include <math.h>

#include "common.cuh"

namespace avsr {

// ------------------------------------------------------------------ embed: x = xs * sqrt(d)   (embedding.py:178)
__global__ void embed_scale_kernel(const float4* __restrict__ xs, float4* __restrict__ x, long n4, float scale) {
  pdl_launch_dependents();
  AVSR_TSPAN_OPEN(130, 0);
  pdl_wait();
  AVSR_TSPAN_DEP();
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    float4 v = xs[i];
    v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
    x[i] = v;
  }
  AVSR_TSPAN_CLOSE();
}

AVSR_TRACE_DEFINE_BIND(trace_bind_elementwise)

int launch_embed_scale(const float* xs, float* x, long n, float scale, cudaStream_t st) {
  AVSR_REQUIRE(n % 4 == 0, "embed: element count %ld not a multiple of 4", n);
  long n4 = n / 4;
  int blocks = (int)((n4 + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  if (blocks < 1) blocks = 1;
  AVSR_LAUNCH(embed_scale_kernel, blocks, 256, 0, st, (const float4*)xs, (float4*)x, n4, scale);
  return AVSR_OK;
}

// ------------------------------------------------------------------ LayerNorm (layer_norm.py:21, eps 1e-12)
// A row (d <= 1024 channels) is held in registers by WPR warps: HBM / L2 sees exactly one read and one write per
// element.  Two-pass mean / centred variance; warp-shuffle reductions, combined across the row's warps through shared
// memory in a fixed order (deterministic).  The r02 launch timeline showed these kernels to be bound by the latency of
// one load -> reduce -> store chain per warp (1 600 warps on 148 SMs is a single, half-empty wave), so more warps per
// row = shorter chains and more loads in flight per SM.  2 warps per row x 4 rows per CTA was best in situ (r02 sweep
// of 1x8, 1x2, 2x4, 2x2, 4x2, 4x1: profiles/r02_ln_sweep.txt).
//   TWO = false : y = LN(x; g1, b1)                                   (y in operand storage or fp32)
//   TWO = true  : y1 = LN(x; g1, b1) (fp32, may alias x) and y = LN(y1; g2, b2) in operand storage -- layer l's
//                 norm_final followed by layer l+1's norm_ff_macaron (conformer_encoder.py:161-162 then :113).
//   NP > 0      : deferred split-K residual update applied while the row is loaded (LnParts): row = x + alpha *
//                 (bias + part[0] + ... + part[NP-1]), fixed order; the updated row is written to pp.x_out when that
//                 is not already the kernel's own fp32 output.  All loads of the row are issued before the first use
//                 and before any store (a store in between would serialise them: possible aliasing).
constexpr int kLnWpr = 2, kLnRpc = 4;   // warps per row, rows per CTA
constexpr int kLnMaxD = 1024;           // 4 float4 per lane at 2 warps per row

__device__ __forceinline__ void ln_named_bar(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// sum over the row's WPR warps; `slot` = this reduction's private shared-memory cells (never reused in the kernel)
template <int WPR>
__device__ __forceinline__ float ln_row_sum(float v, float* slot, int wr, int lane, int bar_id) {
  v = warp_sum(v);
  if constexpr (WPR == 1) return v;
  if (lane == 0) slot[wr] = v;
  ln_named_bar(bar_id, 32 * WPR);
  float t = slot[0];
#pragma unroll
  for (int w = 1; w < WPR; ++w) t += slot[w];
  return t;
}

template <int NP, bool TWO, int WPR, int RPC, int V>   // V = float4 per lane: WPR * 32 * V * 4 >= d
__global__ void __launch_bounds__(32 * WPR * RPC)
ln_kernel(const float* x /* may alias y1 / pp.x_out */, const float* __restrict__ g1, const float* __restrict__ b1,
          const float* __restrict__ g2, const float* __restrict__ b2, float* y1, void* y, int rows, int d,
          int out_kind, LnParts pp) {
  constexpr int STEP = 32 * WPR;                // float4 stride between a lane's vectors
  __shared__ float red[4][RPC][WPR];
  pdl_launch_dependents();
  AVSR_TSPAN_OPEN(TWO ? 110 : 100, NP | (WPR << 8) | (RPC << 12));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rl = warp / WPR, wr = warp - rl * WPR;      // row inside the CTA, warp inside the row
  const int row = blockIdx.x * RPC + rl;
  if (row >= rows) return;                              // whole rows leave together (named barriers are per row)
  const int nvec = d >> 2;
  const int c0 = wr * 32 + lane;
  // parameters are not produced by the previous kernel: fetch them before waiting on it
  float4 gg[V], bb[V], gg2[TWO ? V : 1], bb2[TWO ? V : 1];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = c0 + i * STEP;
    if (c < nvec) {
      gg[i] = reinterpret_cast<const float4*>(g1)[c]; bb[i] = reinterpret_cast<const float4*>(b1)[c];
      if constexpr (TWO) { gg2[i] = reinterpret_cast<const float4*>(g2)[c]; bb2[i] = reinterpret_cast<const float4*>(b2)[c]; }
    }
  }
  float4 pb[NP > 0 ? V : 1];
  if constexpr (NP > 0) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = c0 + i * STEP;
      if (c < nvec) pb[i] = reinterpret_cast<const float4*>(pp.bias)[c];
    }
  }
  pdl_wait();
  AVSR_TSPAN_DEP();
  const long rv = (long)row * nvec;
  const float4* xr = reinterpret_cast<const float4*>(x) + rv;
  float4 v[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int c = c0 + i * STEP;
    if (c < nvec) v[i] = xr[c];
  }
  if constexpr (NP > 0) {
    const float4* p4 = reinterpret_cast<const float4*>(pp.part) + rv;
    const long sv = pp.stride >> 2;
    float4 t[NP][V];
#pragma unroll
    for (int s = 0; s < NP; ++s)
#pragma unroll
      for (int i = 0; i < V; ++i) {
        const int c = c0 + i * STEP;
        if (c < nvec) t[s][i] = p4[s * sv + c];
      }
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float4 a = pb[i];
#pragma unroll
      for (int s = 0; s < NP; ++s) { a.x += t[s][i].x; a.y += t[s][i].y; a.z += t[s][i].z; a.w += t[s][i].w; }
      v[i].x += pp.alpha * a.x; v[i].y += pp.alpha * a.y; v[i].z += pp.alpha * a.z; v[i].w += pp.alpha * a.w;
    }
  }
  const int bar_id = 1 + rl;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (c0 + i * STEP < nvec) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  float mean = ln_row_sum<WPR>(s, red[0][rl], wr, lane, bar_id) / (float)d;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (c0 + i * STEP < nvec) {
      const float a = v[i].x - mean, b = v[i].y - mean, e = v[i].z - mean, f = v[i].w - mean;
      q += (a * a + b * b) + (e * e + f * f);
    }
  float rstd = 1.0f / sqrtf(ln_row_sum<WPR>(q, red[1][rl], wr, lane, bar_id) / (float)d + 1e-12f);
  if constexpr (!TWO) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = c0 + i * STEP;
      if (c < nvec) {
        if (NP > 0 && pp.x_out) reinterpret_cast<float4*>(pp.x_out)[rv + c] = v[i];
        const float4 o = make_float4((v[i].x - mean) * rstd * gg[i].x + bb[i].x, (v[i].y - mean) * rstd * gg[i].y + bb[i].y,
                                     (v[i].z - mean) * rstd * gg[i].z + bb[i].z, (v[i].w - mean) * rstd * gg[i].w + bb[i].w);
        if (y1) reinterpret_cast<float4*>(y1)[rv + c] = o;       // dual output: the fp32 copy (after_norm -> features)
        store_kind4(y, (long)row * d + 4 * c, out_kind, o.x, o.y, o.z, o.w);
      }
    }
  } else {
    float4* y1r = reinterpret_cast<float4*>(y1) + rv;
    s = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = c0 + i * STEP;
      if (c < nvec) {
        v[i].x = (v[i].x - mean) * rstd * gg[i].x + bb[i].x;
        v[i].y = (v[i].y - mean) * rstd * gg[i].y + bb[i].y;
        v[i].z = (v[i].z - mean) * rstd * gg[i].z + bb[i].z;
        v[i].w = (v[i].w - mean) * rstd * gg[i].w + bb[i].w;
        y1r[c] = v[i];
        s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
      }
    }
    mean = ln_row_sum<WPR>(s, red[2][rl], wr, lane, bar_id) / (float)d;
    q = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i)
      if (c0 + i * STEP < nvec) {
        const float a = v[i].x - mean, b = v[i].y - mean, e = v[i].z - mean, f = v[i].w - mean;
        q += (a * a + b * b) + (e * e + f * f);
      }
    rstd = 1.0f / sqrtf(ln_row_sum<WPR>(q, red[3][rl], wr, lane, bar_id) / (float)d + 1e-12f);
#pragma unroll
    for (int i = 0; i < V; ++i) {
      const int c = c0 + i * STEP;
      if (c < nvec)
        store_kind4(y, (long)row * d + 4 * c, out_kind, (v[i].x - mean) * rstd * gg2[i].x + bb2[i].x,
                    (v[i].y - mean) * rstd * gg2[i].y + bb2[i].y, (v[i].z - mean) * rstd * gg2[i].z + bb2[i].z,
                    (v[i].w - mean) * rstd * gg2[i].w + bb2[i].w);
    }
  }
  AVSR_TSPAN_CLOSE();
}

template <int NP, bool TWO>
static int launch_ln_np(const float* x, const float* g1, const float* b1, const float* g2, const float* b2, float* y1,
                        void* y, int rows, int d, int out_kind, cudaStream_t st, const LnParts& pp) {
  // vectors per lane: 3 for the reference's d = 768, 4 up to 1024 channels
  if (d <= 768)
    AVSR_LAUNCH((ln_kernel<NP, TWO, kLnWpr, kLnRpc, 3>), cdiv(rows, kLnRpc), 32 * kLnWpr * kLnRpc, 0, st, x, g1, b1, g2,
                b2, y1, y, rows, d, out_kind, pp);
  else
    AVSR_LAUNCH((ln_kernel<NP, TWO, kLnWpr, kLnRpc, 4>), cdiv(rows, kLnRpc), 32 * kLnWpr * kLnRpc, 0, st, x, g1, b1, g2,
                b2, y1, y, rows, d, out_kind, pp);
  return AVSR_OK;
}

template <bool TWO>
static int launch_ln(const float* x, const float* g1, const float* b1, const float* g2, const float* b2, float* y1,
                     void* y, int rows, int d, int out_kind, cudaStream_t st, const LnParts* parts) {
  AVSR_REQUIRE(d % 4 == 0 && d <= kLnMaxD && d > 0, "layernorm: d=%d must be a multiple of 4 and <= %d", d, kLnMaxD);
  if (rows <= 0) return AVSR_OK;
  const LnParts pp = parts ? *parts : LnParts{};
  switch (pp.nparts) {
    case 0: return launch_ln_np<0, TWO>(x, g1, b1, g2, b2, y1, y, rows, d, out_kind, st, pp);
    case kW2Splits: return launch_ln_np<kW2Splits, TWO>(x, g1, b1, g2, b2, y1, y, rows, d, out_kind, st, pp);
    default: AVSR_REQUIRE(false, "layernorm: %d k-slices not instantiated (0, %d)", pp.nparts, kW2Splits);
  }
  return AVSR_OK;
}

int launch_layernorm2(const float* x, const float* g1, const float* b1, const float* g2, const float* b2, float* y1,
                      void* y2, int rows, int d, int out_kind, cudaStream_t st, const LnParts* parts) {
  return launch_ln<true>(x, g1, b1, g2, b2, y1, y2, rows, d, out_kind, st, parts);
}

int launch_layernorm(const float* x, const float* g, const float* b, void* y, int rows, int d, int out_kind,
                     cudaStream_t st, const LnParts* parts) {
  return launch_ln<false>(x, g, b, nullptr, nullptr, nullptr, y, rows, d, out_kind, st, parts);
}

int launch_layernorm_dual(const float* x, const float* g, const float* b, float* y_f32, void* y_op, int rows, int d,
                          int out_kind, cudaStream_t st) {
  return launch_ln<false>(x, g, b, nullptr, nullptr, y_f32, y_op, rows, d, out_kind, st, nullptr);
}

// ------------------------------------------------------------------ rel-pos sinusoid table (embedding.py:139-184)
// Row m <-> rel = T-1-m; even channels sin(rel*w_i), odd channels cos(rel*w_i), w_i = exp(2i * -(ln 1e4 / d)).
// The reference evaluates everything in fp32: the frequency is a correctly rounded fp32 exp, the
// argument an fp32 product; sinf/cosf here take the full-range (non fast-math) path.
__global__ void sinusoid_kernel(void* __restrict__ pe, int T, int d, int out_kind) {
  pdl_launch_dependents();
  AVSR_TSPAN_OPEN(140, 0);
  pdl_wait();
  AVSR_TSPAN_DEP();
  const int half = d >> 1;
  const long total = (long)(2 * T - 1) * half;
  const float step = (float)(-(log(10000.0) / (double)d));
  for (long i = blockIdx.x * (long)blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
    const int m = (int)(i / half), c = (int)(i - (long)m * half);
    const float e = (float)(2 * c) * step;
    const float inv = (float)exp((double)e);
    const int rel = T - 1 - m;
    float arg = fabsf((float)rel) * inv;
    if (rel < 0) arg = -arg;
    const float s = sinf(arg), co = cosf(arg);
    const long idx = (long)m * d + 2 * c;
    if (out_kind == OP_F16) {
      *reinterpret_cast<__half2*>(reinterpret_cast<__half*>(pe) + idx) = __halves2half2(to_half_sat(s), to_half_sat(co));
    } else if (out_kind == OP_TF32) {
      *reinterpret_cast<float2*>(reinterpret_cast<float*>(pe) + idx) = make_float2(round_tf32(s), round_tf32(co));
    } else {
      *reinterpret_cast<float2*>(reinterpret_cast<float*>(pe) + idx) = make_float2(s, co);
    }
  }
  AVSR_TSPAN_CLOSE();
}

int launch_sinusoid(void* pe, int T, int d, int out_kind, cudaStream_t st) {
  AVSR_REQUIRE(T > 0 && d > 0 && d % 2 == 0, "sinusoid: bad T=%d d=%d", T, d);
  const long total = (long)(2 * T - 1) * (d / 2);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  AVSR_LAUNCH(sinusoid_kernel, blocks, 256, 0, st, pe, T, d, out_kind);
  return AVSR_OK;
}

// ------------------------------------------------------------------ depthwise conv + BN(eval) + SiLU
// y[b,t,c] = silu( (sum_k wt[k][c] * x[b, t+k-half, c]) * scale[c] + shift[c] ),  x zero outside [0,T) per
// utterance row b -- no length mask: padded frames are data (conformer_encoder.py:30-35, SURVEY.md D6).
// scale/shift fold the depthwise bias and the BatchNorm running statistics (avsr_prepare_weights).
// Tile: CH channels x 64 frames per CTA; the (64+K-1) x CH input patch and the K x CH taps are staged
// in shared memory with coalesced float4 loads along the channel axis.  Each thread produces 8 consecutive frames of
// one channel quad with a register sliding window: per tap ONE new input row and one tap vector are read from
// shared memory for 8 outputs (the v1 kernel read 2 per output pair: 4x more shared-memory traffic, r01 profile).
constexpr int kDwTT = 64;    // frames per CTA
constexpr int kDwFr = 8;     // frames per thread
// channels per CTA (CH): 32 for K = 31 (8 quads, 64 threads, 672 CTAs at S2: the same halo ratio as 64 and full
// 128-byte row segments, with twice as many CTAs in flight per SM to hide the load -> barrier -> compute -> store chain
// of each); 64 for the runtime-K kernel

template <int K, int QPR>
__device__ __forceinline__ void dw_accumulate(const float4* in_s, const float4* w_s, int q, int ts, int k_runtime,
                                              float4 (&acc)[kDwFr]) {
  // K > 0: fully unrolled (window shifts become register renames); K == 0: runtime tap count
  constexpr int KK = K > 0 ? K : 1;
  float4 win[kDwFr];
#pragma unroll
  for (int j = 0; j < kDwFr - 1; ++j) win[j + 1] = in_s[(ts * kDwFr + j) * QPR + q];
  const int taps = K > 0 ? KK : k_runtime;
#pragma unroll
  for (int k = 0; k < (K > 0 ? KK : 256); ++k) {
    if (K == 0 && k >= taps) break;
#pragma unroll
    for (int j = 0; j < kDwFr - 1; ++j) win[j] = win[j + 1];
    win[kDwFr - 1] = in_s[(ts * kDwFr + kDwFr - 1 + k) * QPR + q];
    const float4 w = w_s[k * QPR + q];
#pragma unroll
    for (int j = 0; j < kDwFr; ++j) {
      acc[j].x = fmaf(w.x, win[j].x, acc[j].x); acc[j].y = fmaf(w.y, win[j].y, acc[j].y);
      acc[j].z = fmaf(w.z, win[j].z, acc[j].z); acc[j].w = fmaf(w.w, win[j].w, acc[j].w);
    }
  }
}

template <int K, int CH>
__global__ void __launch_bounds__((CH / 4) * (kDwTT / kDwFr))
dwconv_bn_silu_kernel(const float* __restrict__ x, const float* __restrict__ wt, const float* __restrict__ scale,
                      const float* __restrict__ shift, void* __restrict__ y, int T, int C, int k_runtime, int out_kind) {
  constexpr int QPR = CH / 4;                                // float4 quads per staged row
  constexpr int NT = QPR * (kDwTT / kDwFr);                  // threads per CTA
  extern __shared__ float4 dw_smem[];
  pdl_launch_dependents();
  AVSR_TSPAN_OPEN(120, CH);
  const int Kt = K > 0 ? K : k_runtime;
  const int rows_in = kDwTT + Kt - 1;
  float4* in_s = dw_smem;                          // [rows_in][QPR]
  float4* w_s = dw_smem + rows_in * QPR;           // [K][QPR]
  const int c0 = blockIdx.x * CH;
  const int t0 = blockIdx.y * kDwTT;
  const int b = blockIdx.z;
  const int half = (Kt - 1) >> 1;
  const int tid = threadIdx.x;
  const float* xb = x + (long)b * T * C;

  // the taps are parameters: stage them before waiting on the producer of x
  for (int i = tid; i < Kt * QPR; i += NT) {
    const int k = i / QPR, q = i % QPR;
    const int c = c0 + q * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C) v = *reinterpret_cast<const float4*>(wt + (long)k * C + c);
    w_s[i] = v;
  }
  pdl_wait();
  AVSR_TSPAN_DEP();
  {
    const int total = rows_in * QPR;
    for (int i0 = tid; i0 < total; i0 += 4 * NT) {   // 4 independent 16-byte loads in flight per thread
      float4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * NT;
        const int r = i / QPR, q = i % QPR;
        const int t = t0 - half + r, c = c0 + q * 4;
        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < total && t >= 0 && t < T && c < C) v[u] = *reinterpret_cast<const float4*>(xb + (long)t * C + c);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = i0 + u * NT;
        if (i < total) in_s[i] = v[u];
      }
    }
  }
  __syncthreads();

  const int q = tid % QPR, ts = tid / QPR;         // channel quad, group of 8 frames
  const int c = c0 + q * 4;
  if (c >= C) return;
  float4 acc[kDwFr];
#pragma unroll
  for (int j = 0; j < kDwFr; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  dw_accumulate<K, QPR>(in_s, w_s, q, ts, k_runtime, acc);
  const float4 sc = *reinterpret_cast<const float4*>(scale + c);
  const float4 sh = *reinterpret_cast<const float4*>(shift + c);
#pragma unroll
  for (int j = 0; j < kDwFr; ++j) {
    const int t = t0 + ts * kDwFr + j;
    if (t >= T) break;
    float4 o;
    o.x = fmaf(acc[j].x, sc.x, sh.x); o.y = fmaf(acc[j].y, sc.y, sh.y);
    o.z = fmaf(acc[j].z, sc.z, sh.z); o.w = fmaf(acc[j].w, sc.w, sh.w);
    if (out_kind < 0) {         // raw fp32 (training path: plain conv + bias, or the input-gradient correlation)
    } else if (out_kind == OP_F32) {   // exact path for the fp32 reference mode
      o.x *= sigmoidf_acc(o.x); o.y *= sigmoidf_acc(o.y); o.z *= sigmoidf_acc(o.z); o.w *= sigmoidf_acc(o.w);
    } else {
      o.x *= sigmoidf_fast(o.x); o.y *= sigmoidf_fast(o.y); o.z *= sigmoidf_fast(o.z); o.w *= sigmoidf_fast(o.w);
    }
    store_kind4(y, ((long)b * T + t) * C + c, out_kind, o.x, o.y, o.z, o.w);
  }
  AVSR_TSPAN_CLOSE();
}

template <int K, int CH>
static int launch_dw(const float* x, const float* wt, const float* scale, const float* shift, void* y, int B, int T, int C, int Kr,
                     int out_kind, cudaStream_t st) {
  const size_t smem = (size_t)(kDwTT + Kr - 1 + Kr) * (CH / 4) * sizeof(float4);
  dim3 grid(cdiv(C, CH), cdiv(T, kDwTT), B);
  if (smem > 48 * 1024)
    AVSR_CUDA_TRY(cudaFuncSetAttribute((dwconv_bn_silu_kernel<K, CH>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  AVSR_LAUNCH((dwconv_bn_silu_kernel<K, CH>), grid, (CH / 4) * (kDwTT / kDwFr), smem, st, x, wt, scale, shift, y, T, C, Kr, out_kind);
  return AVSR_OK;
}

int launch_dwconv_bn_silu(const float* x, const float* wt, const float* scale, const float* shift, void* y, int B,
                          int T, int C, int K, int out_kind, cudaStream_t st) {
  AVSR_REQUIRE(C % 4 == 0 && K % 2 == 1 && K >= 1 && K <= 255, "dwconv: C=%d must be a multiple of 4, K=%d odd", C, K);
  if (B <= 0 || T <= 0) return AVSR_OK;
  if (K == 31)   // the reference's cnn_module_kernel (e2e_asr_conformer.py:38): fully unrolled taps
    return launch_dw<31, 32>(x, wt, scale, shift, y, B, T, C, K, out_kind, st);
  return launch_dw<0, 64>(x, wt, scale, shift, y, B, T, C, K, out_kind, st);
}

}  // namespace avsr
