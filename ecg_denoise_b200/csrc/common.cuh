// common.cuh -- shared device helpers for the RA-LENet sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "ralenet_b200.h"

#ifndef RL_NT
#define RL_NT 256          // threads per CTA (a translation unit may define it before including this header)
#endif
#ifndef RL_MINB
#define RL_MINB 1          // min CTAs per SM hint for __launch_bounds__
#endif
#ifndef RL_FW_MAXC
#define RL_FW_MAXC 16      // stages with C <= this accumulate their weight gradients inside the data-gradient kernels
#endif
#define RL_HD 4            // head dim (model/transformer.py:277: dim // num_heads == 4 at every stage)
#define RL_LOG2E 1.4426950408889634f
#define RL_LN_EPS 1e-5f

// phase timestamps (debug builds only, -DRL_TRACE): RL_TRACE_DEFINE(tag) once per translation unit, then
// RL_TS(tag, i) stores the SM clock of thread 0 into slot i < 16 of this CTA; read with ralenet_debug_trace_read_<tag>
#ifdef RL_TRACE
#define RL_TRACE_DEFINE(tag)                                                          \
  __device__ long long g_trace_##tag[4096 * 16];                                      \
  extern "C" int ralenet_debug_trace_read_##tag(long long* out, int n) {              \
    return (int)cudaMemcpyFromSymbol(out, g_trace_##tag, sizeof(long long) * n);      \
  }
#define RL_TS(tag, i) do { if (threadIdx.x == 0 && blockIdx.x < 4096) g_trace_##tag[blockIdx.x * 16 + (i)] = clock64(); } while (0)
#else
#define RL_TRACE_DEFINE(tag)
#define RL_TS(tag, i) do { } while (0)
#endif

void rl_set_error(const char* fmt, ...);
void rl_count_launch();
// profiler label "what<tag0,tag1>suffix" (suffix ":tf32" marks the single-pass TF32 forward kernels)
int rl_check_launch(const char* what, int tag0 = -1, int tag1 = -1, const char* suffix = "");
constexpr const char* rl_tf32_tag(bool tf32) { return tf32 ? ":tf32" : ""; }
void rl_prof_pre(cudaStream_t st);     // profiling: event right before the next launch on the profiled stream

#define RL_REQUIRE(cond, code, ...)            \
  do {                                         \
    if (!(cond)) {                             \
      rl_set_error(__VA_ARGS__);               \
      return (code);                           \
    }                                          \
  } while (0)

// Programmatic dependent launch: the kernel may be scheduled while the previous kernel on the stream drains;
// it must call pdl_wait() before touching global memory.  Captured into CUDA graphs as programmatic edges.
// cluster > 0: consecutive groups of `cluster` CTAs along x form a thread-block cluster (distributed shared memory).
template <typename... KArgs, typename... Args>
static inline void rl_launch_pdl_cluster(int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                                         cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster > 0) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[n].val.programmaticStreamSerializationAllowed = 1;
  ++n;
  cfg.attrs = attr;
  cfg.numAttrs = n;
  rl_prof_pre(st);
  cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);      // errors surface through rl_check_launch()
}
template <typename... KArgs, typename... Args>
static inline void rl_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                 Args... args) {
  rl_launch_pdl_cluster(0, kernel, grid, block, smem, st, args...);
}
// L2 prefetch of tensors that were saved by the forward pass (they sit in HBM by the time the backward reads them):
// issued before griddepcontrol.wait, the HBM latency passes behind the tail of the preceding kernel and the loads of
// the kernel proper hit L2.  A hint: no register, no dependency, nothing to wait for.
__device__ __forceinline__ void prefetch_l2(const void* p) {
#ifndef RL_NO_L2_PREFETCH      // A/B builds; measured on the graphed step: 2.229 ms without, 2.212 ms with
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
#endif
}
// `bytes` from p (128-byte lines), spread over the threads of the CTA
__device__ __forceinline__ void prefetch_l2_block(const void* p, int bytes) {
  for (int o = threadIdx.x * 128; o < bytes; o += RL_NT * 128) prefetch_l2(reinterpret_cast<const char*>(p) + o);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// SplitMix64 finaliser: the counter-based hash behind the device-side batch sources (synth.cu, records.cu)
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

template <typename K>
static inline int rl_set_smem(K kernel, size_t bytes) {
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) {
    rl_set_error("cudaFuncSetAttribute(%zu B smem): %s", bytes, cudaGetErrorString(e));
    return RL_ERR_CUDA;
  }
  return RL_OK;
}

// ---------------------------------------------------------------------------------------------
// nn.GELU() (exact erf form, x * Phi(x)) without the branchy libdevice erff: Abramowitz-Stegun 7.1.26,
//   1 - erf(z) = (a1 t + ... + a5 t^5) exp(-z^2),  t = 1 / (1 + p z),  z = |x| / sqrt(2)   (|error| <= 1.5e-7),
// evaluated as the TAIL q = (1 - erf(z)) / 2, so that Phi(x) = q for x < 0 carries no cancellation.  Against the
// fp64 GELU the fp32 result is as close as the erff-based one (4.6e-7 vs 4.5e-7 absolute on [-12, 12], checked
// in tests/test_cpu_host.py) at a third of the instructions; the exponential doubles as the Gaussian of GELU'.
__device__ __forceinline__ void gelu_parts(float x, float& cdf, float& gauss /* exp(-x^2 / 2) */) {
  const float z = fabsf(x) * 0.70710678118654752f;
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, z, 1.0f)));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -0.72134752044448170f));      // exp(-x^2 / 2)
  float q = fmaf(0.5f * 1.061405429f, t, 0.5f * -1.453152027f);
  q = fmaf(q, t, 0.5f * 1.421413741f);
  q = fmaf(q, t, 0.5f * -0.284496736f);
  q = fmaf(q, t, 0.5f * 0.254829592f);
  q = q * t * e;                                    // (1 - erf(z)) / 2
  cdf = (x < 0.f) ? q : 1.0f - q;
  gauss = e;
}
__device__ __forceinline__ float gelu_f(float x) {
  float cdf, e;
  gelu_parts(x, cdf, e);
  return x * cdf;
}
__device__ __forceinline__ float gelu_grad_f(float x) {
  float cdf, e;
  gelu_parts(x, cdf, e);
  return fmaf(x * e, 0.3989422804014327f, cdf);
}

// gelu(x) and gelu'(x) sharing one evaluation
__device__ __forceinline__ void gelu_both(float x, float& g, float& dg) {
  float cdf, e;
  gelu_parts(x, cdf, e);
  g = x * cdf;
  dg = fmaf(x * e, 0.3989422804014327f, cdf);
}

// ---- two GELUs at once on Blackwell's packed fp32 pipe (FMUL2 / FFMA2 / FADD2): same arithmetic, same bits, as two
// gelu_parts() calls, two thirds of the issue slots.  GELU and GELU' are ~15 % of all instructions of a training step
// (2 + 2 evaluations per hidden element and block).
__device__ __forceinline__ void pk_mul(float x0, float x1, float y0, float y1, float& r0, float& r1) {
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmul.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(y0), "f"(y1));
}
__device__ __forceinline__ void pk_fma(float x0, float x1, float y0, float y1, float z0, float z1, float& r0, float& r1) {
  asm("{\n\t.reg .b64 a, b, c, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmov.b64 c, {%6, %7};\n\t"
      "fma.rn.f32x2 d, a, b, c;\n\tmov.b64 {%0, %1}, d;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(y0), "f"(y1), "f"(z0), "f"(z1));
}
__device__ __forceinline__ void gelu_parts2(float x0, float x1, float& cdf0, float& cdf1, float& g0, float& g1) {
  float z0, z1, u0, u1, t0, t1, s0, s1, e0, e1, q0, q1;
  pk_mul(fabsf(x0), fabsf(x1), 0.70710678118654752f, 0.70710678118654752f, z0, z1);
  pk_fma(z0, z1, 0.3275911f, 0.3275911f, 1.0f, 1.0f, u0, u1);
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t0) : "f"(u0));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t1) : "f"(u1));
  pk_mul(x0, x1, x0, x1, s0, s1);
  pk_mul(s0, s1, -0.72134752044448170f, -0.72134752044448170f, s0, s1);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(s0));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(s1));
  pk_fma(t0, t1, 0.5f * 1.061405429f, 0.5f * 1.061405429f, 0.5f * -1.453152027f, 0.5f * -1.453152027f, q0, q1);
  pk_fma(q0, q1, t0, t1, 0.5f * 1.421413741f, 0.5f * 1.421413741f, q0, q1);
  pk_fma(q0, q1, t0, t1, 0.5f * -0.284496736f, 0.5f * -0.284496736f, q0, q1);
  pk_fma(q0, q1, t0, t1, 0.5f * 0.254829592f, 0.5f * 0.254829592f, q0, q1);
  pk_mul(q0, q1, t0, t1, q0, q1);
  pk_mul(q0, q1, e0, e1, q0, q1);
  cdf0 = (x0 < 0.f) ? q0 : 1.0f - q0;
  cdf1 = (x1 < 0.f) ? q1 : 1.0f - q1;
  g0 = e0;
  g1 = e1;
}
__device__ __forceinline__ void gelu2(float x0, float x1, float& y0, float& y1) {
  float c0, c1, e0, e1;
  gelu_parts2(x0, x1, c0, c1, e0, e1);
  pk_mul(x0, x1, c0, c1, y0, y1);
}
// gelu and gelu' of two values sharing one evaluation each
__device__ __forceinline__ void gelu_both2(float x0, float x1, float& g0, float& g1, float& d0, float& d1) {
  float c0, c1, e0, e1, w0, w1;
  gelu_parts2(x0, x1, c0, c1, e0, e1);
  pk_mul(x0, x1, c0, c1, g0, g1);
  pk_mul(x0, x1, e0, e1, w0, w1);
  pk_fma(w0, w1, 0.3989422804014327f, 0.3989422804014327f, c0, c1, d0, d1);
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 fma4(float4 a, float4 b, float4 c) {
  return make_float4(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z), fmaf(a.w, b.w, c.w));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <int GS>
__device__ __forceinline__ float group_sum(float v) {        // sum over aligned groups of GS lanes
#pragma unroll
  for (int o = GS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// block-wide sum of `v` (all RL_NT threads must call); result valid in every thread.
__device__ __forceinline__ float block_sum(float v, float* s_red /* >= 32 floats */) {
  v = warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[w] = v;
  __syncthreads();
  float r = (lane < (RL_NT >> 5)) ? s_red[lane] : 0.f;
  r = warp_sum(r);
  return r;
}

// ---------------------------------------------------------------------------------------------
// Register-tiled SIMT micro GEMM on shared-memory operands:
//   acc[i][j] += sum_k A[(m0+i)*sam + k*sak] * B[k*sbk + n0 + j*nst]
template <int RM, int RN>
__device__ __forceinline__ void micro_gemm(float (&acc)[RM][RN], const float* __restrict__ A, int sam, int sak,
                                           const float* __restrict__ B, int sbk, int m0, int n0, int nst, int K) {
  const float* a_base = A + m0 * sam;
  const float* b_base = B + n0;
#pragma unroll 4
  for (int k = 0; k < K; ++k) {
    float a[RM], b[RN];
#pragma unroll
    for (int i = 0; i < RM; ++i) a[i] = a_base[i * sam + k * sak];
#pragma unroll
    for (int j = 0; j < RN; ++j) b[j] = b_base[k * sbk + j * nst];
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < RN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
  }
}

// ---------------------------------------------------------------------------------------------
// Parameter-gradient output of a backward kernel.  Default: fp32 atomics into the gradient, so the low bits depend on
// the order in which CTAs arrive.  Deterministic mode (DET, RL_NET_DETERMINISTIC): the gradient pointer handed to the
// kernel is a partial slab [slots][n] (rl_det_take), every slot is written by exactly one CTA with plain stores, and
// rl_launch_grad_reduce() later adds the slots up in slot order.  grad_slot() moves a slab pointer to the slot of the
// calling CTA; the slot is a function of the work item only (window, tile, token slice), never of timing.
template <bool DET>
__device__ __forceinline__ void grad_add(float* p, float v) {
  if constexpr (DET) *p = v;
  else atomicAdd(p, v);
}
template <bool DET>
__device__ __forceinline__ float* grad_slot(float* p, size_t n, int slot) {
  return (DET && p != nullptr) ? p + (size_t)slot * n : p;
}

// ---------------------------------------------------------------------------------------------
// LayerNorm over C channels of `rows` tokens (eps 1e-5, biased variance, like nn.LayerNorm).
// A group of GS = min(C,32) lanes owns one token; each lane holds CPL = C/GS channels.
// load(t, c) returns the pre-norm value; store(t, c, zhat, rstd_is_unused) receives zhat.
// (Round 2 gave every lane ONE channel at C <= 32: 16 lanes per token at C = 16, four trips over the 128 tokens with
// four 4-step shuffle reductions each.  Four consecutive channels per lane make it one trip with 2-step reductions:
// a quarter of the shuffles, rsqrt and loop overhead -- the LayerNorm phases were 6 - 10 % of the narrow kernels.)
template <int C>
struct LnGeom {
  static_assert(C % 4 == 0 && C / 4 <= 32, "LnGeom: 8 <= C <= 128, C % 4 == 0");
  static constexpr int CPL = 4;                       // consecutive channels per lane
  static constexpr int GS = C / CPL;                  // lanes per token
  static constexpr int TPW = 32 / GS;                 // tokens per warp per iteration
  static constexpr int TPI = TPW * (RL_NT / 32);      // tokens per CTA iteration (TPI * C = 2048: one trip per window)
};

// float4 form: load4(t, c) returns the pre-norm values of channels c..c+3 (c % 4 == 0) of token t, store4(t, c, zhat4)
// receives their normalised values -- one 16-byte access per lane where the caller's arrays allow it
template <int C, class Load4, class Store4>
__device__ __forceinline__ void ln_forward_rows4(int rows, Load4 load4, Store4 store4) {
  using G = LnGeom<C>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane % G::GS, gi = lane / G::GS;
  // unrolled (rows is a compile-time constant at the call sites) so that the global loads of every trip are in flight
  // together instead of one L2 round trip per trip
#pragma unroll
  for (int t0 = 0; t0 < rows; t0 += G::TPI) {
    const int t = t0 + warp * G::TPW + gi;
    const bool ok = t < rows;
    float4 z = ok ? load4(t, 4 * gl) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float mu = group_sum<G::GS>((z.x + z.y) + (z.z + z.w)) * (1.0f / C);
    z.x -= mu; z.y -= mu; z.z -= mu; z.w -= mu;
    const float rstd = rsqrtf(group_sum<G::GS>((z.x * z.x + z.y * z.y) + (z.z * z.z + z.w * z.w)) * (1.0f / C) + RL_LN_EPS);
    if (ok) store4(t, 4 * gl, make_float4(z.x * rstd, z.y * rstd, z.z * rstd, z.w * rstd));
  }
}
// element form: load(t, c) / store(t, c, zhat)
template <int C, class Load, class Store>
__device__ __forceinline__ void ln_forward_rows(int rows, Load load, Store store) {
  ln_forward_rows4<C>(
      rows, [&](int t, int c) { return make_float4(load(t, c), load(t, c + 1), load(t, c + 2), load(t, c + 3)); },
      [&](int t, int c, float4 zh) {
        store(t, c, zh.x); store(t, c + 1, zh.y); store(t, c + 2, zh.z); store(t, c + 3, zh.w);
      });
}

// LayerNorm backward for `rows` tokens.
//   loadz4(t,c): pre-norm input of channels c..c+3;  loaddu4(t,c): gradient w.r.t. the LN output;  gamma: [C]
//   emit4(t, c, dz4, zhat4): receives the gradient w.r.t. the pre-norm input and zhat
//   dgam/dbet partial sums are accumulated into s_gb[0:C] / s_gb[C:2C] (shared, pre-zeroed) with atomics.
//   WP = true: s_gb is [RL_NT/32][2C], one row of partial sums per WARP written with plain stores (no pre-zeroing, no
//   shared-memory atomics: those are compare-and-swap loops for fp32 and 16 warps x TPW token groups contend for every
//   word -- 8 % of the samples of the narrow backward kernels, ncu r2_v32); ln_backward_finish() adds the rows up.
template <int C, bool WP = false, class LoadZ4, class LoadDu4, class Emit4>
__device__ __forceinline__ void ln_backward_rows4(int rows, const float* __restrict__ gamma, float* s_gb, LoadZ4 loadz4,
                                                  LoadDu4 loaddu4, Emit4 emit4) {
  using G = LnGeom<C>;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gl = lane % G::GS, gi = lane / G::GS;
  float gam[4], ag[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f};
  {
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(gamma) + gl);
    gam[0] = g4.x; gam[1] = g4.y; gam[2] = g4.z; gam[3] = g4.w;
  }
#pragma unroll
  for (int t0 = 0; t0 < rows; t0 += G::TPI) {
    const int t = t0 + warp * G::TPW + gi;
    const bool ok = t < rows;
    float z[4] = {0.f, 0.f, 0.f, 0.f}, du[4] = {0.f, 0.f, 0.f, 0.f};
    if (ok) {
      const float4 z4 = loadz4(t, 4 * gl), d4 = loaddu4(t, 4 * gl);
      z[0] = z4.x; z[1] = z4.y; z[2] = z4.z; z[3] = z4.w;
      du[0] = d4.x; du[1] = d4.y; du[2] = d4.z; du[3] = d4.w;
    }
    const float mu = group_sum<G::GS>((z[0] + z[1]) + (z[2] + z[3])) * (1.0f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      z[i] -= mu;
      q += z[i] * z[i];
    }
    const float rstd = rsqrtf(group_sum<G::GS>(q) * (1.0f / C) + RL_LN_EPS);
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      z[i] *= rstd;                       // zhat
      ag[i] += du[i] * z[i];
      ab[i] += du[i];
      du[i] *= gam[i];                    // dzhat
      s1 += du[i];
      s2 += du[i] * z[i];
    }
    s1 = group_sum<G::GS>(s1) * (1.0f / C);
    s2 = group_sum<G::GS>(s2) * (1.0f / C);
    if (ok)
      emit4(t, 4 * gl,
            make_float4(rstd * (du[0] - s1 - z[0] * s2), rstd * (du[1] - s1 - z[1] * s2), rstd * (du[2] - s1 - z[2] * s2),
                        rstd * (du[3] - s1 - z[3] * s2)),
            make_float4(z[0], z[1], z[2], z[3]));
  }
  if (WP) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
#pragma unroll
      for (int o = G::GS; o < 32; o <<= 1) {            // the TPW token groups of this warp hold the same channels
        ag[i] += __shfl_xor_sync(0xffffffffu, ag[i], o);
        ab[i] += __shfl_xor_sync(0xffffffffu, ab[i], o);
      }
    }
    if (gi == 0) {
      *reinterpret_cast<float4*>(s_gb + warp * 2 * C + 4 * gl) = make_float4(ag[0], ag[1], ag[2], ag[3]);
      *reinterpret_cast<float4*>(s_gb + warp * 2 * C + C + 4 * gl) = make_float4(ab[0], ab[1], ab[2], ab[3]);
    }
  } else if (s_gb != nullptr) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      atomicAdd(&s_gb[4 * gl + i], ag[i]);
      atomicAdd(&s_gb[C + 4 * gl + i], ab[i]);
    }
  }
}
// element form: loadz(t,c), loaddu(t,c), emit(t, c, dz, zhat)
template <int C, bool WP = false, class LoadZ, class LoadDu, class Emit>
__device__ __forceinline__ void ln_backward_rows(int rows, const float* __restrict__ gamma, float* s_gb, LoadZ loadz,
                                                 LoadDu loaddu, Emit emit) {
  ln_backward_rows4<C, WP>(
      rows, gamma, s_gb,
      [&](int t, int c) { return make_float4(loadz(t, c), loadz(t, c + 1), loadz(t, c + 2), loadz(t, c + 3)); },
      [&](int t, int c) { return make_float4(loaddu(t, c), loaddu(t, c + 1), loaddu(t, c + 2), loaddu(t, c + 3)); },
      [&](int t, int c, float4 dz, float4 zh) {
        emit(t, c, dz.x, zh.x); emit(t, c + 1, dz.y, zh.y); emit(t, c + 2, dz.z, zh.z); emit(t, c + 3, dz.w, zh.w);
      });
}
// after a CTA barrier behind ln_backward_rows<C, true>: d_ln_w / d_ln_b += the per-warp partial rows
// (DET: d_ln_w / d_ln_b are this CTA's slots of partial slabs, see grad_add)
template <int C, bool DET = false>
__device__ __forceinline__ void ln_backward_finish(const float* s_part, float* __restrict__ d_ln_w,
                                                   float* __restrict__ d_ln_b) {
  if (d_ln_w == nullptr) return;
  for (int i = threadIdx.x; i < 2 * C; i += RL_NT) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < RL_NT / 32; ++w) s += s_part[w * 2 * C + i];
    grad_add<DET>((i < C) ? d_ln_w + i : d_ln_b + i - C, s);
  }
}

// ---------------------------------------------------------------------------------------------
// Tensor-core CTA GEMM on shared-memory operands: legacy mma.sync m16n8k8 TF32 with the 3xTF32 split
// (a = a_hi + a_lo, D += a_lo*b_hi + a_hi*b_lo + a_hi*b_hi), which keeps fp32-grade accuracy
// (the north star's 1e-3 tolerance leaves no room for single-pass TF32 through 18 blocks).
// Measured on this B200 (profiles/mma_rate_b200.txt): mma.sync TF32 277 TFLOP/s vs FFMA 72 TFLOP/s.
//
// out[M x N] is spread over the 8 warps; each warp owns RT x CT m16n8 tiles.  Operand layouts:
//   A_MK: A(m,k) at A[m*lda + k]  (conflict-free when lda % 8 == 4)    A_KM: A[k*lda + m]  (lda % 32 in {8,24})
//   B_NK: B(k,n) at B[n*ldb + k]  (ldb % 8 == 4)                       B_KN: B[k*ldb + n]  (ldb % 32 in {8,24})
enum { A_MK = 0, A_KM = 1 };
enum { B_NK = 0, B_KN = 1 };

__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// single-pass TF32 operand (RL_F_TF32): x rounded to nearest (ties away) to a 10-bit mantissa.  Rounding, not the
// truncation of split_tf32, so that the errors of a long contraction (fc2: 4C = 512 terms) do not all lean one way.
__device__ __forceinline__ uint32_t rna_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// x = hi + lo exactly; hi has a 10-bit mantissa (truncated), lo is fed as is (the MMA ignores its low 13 bits)
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// Blackwell packed fp32 arithmetic on register pairs (SASS FADD2 / FMUL2): one issue slot for two lanes of work
__device__ __forceinline__ void sub_f32x2(float x0, float x1, float y0, float y1, float& r0, float& r1) {
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tsub.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(y0), "f"(y1));
}
__device__ __forceinline__ void add_f32x2(float x0, float x1, float y0, float y1, float& r0, float& r1) {
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tadd.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(y0), "f"(y1));
}
__device__ __forceinline__ void mul_f32x2(float x0, float x1, float y0, float y1, float& r0, float& r1) {
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmul.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(y0), "f"(y1));
}
// two splits at once: the remainders come from ONE packed subtraction (Blackwell `sub.f32x2`, SASS FADD2) -- the split
// arithmetic is 18 % of the instructions of the narrow-stage GEMM kernels (ncu r2_v24), this takes a quarter of it out
__device__ __forceinline__ void split_tf32x2(float x0, float x1, uint32_t& h0, uint32_t& h1, uint32_t& l0, uint32_t& l1) {
  h0 = __float_as_uint(x0) & 0xffffe000u;
  h1 = __float_as_uint(x1) & 0xffffe000u;
  float r0, r1;
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tsub.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r0), "=f"(r1)
      : "f"(x0), "f"(x1), "f"(__uint_as_float(h0)), "f"(__uint_as_float(h1)));
  l0 = __float_as_uint(r0);
  l1 = __float_as_uint(r1);
}

template <int M, int N>
struct MmaTile {
  static constexpr int MT = M / 16, NT = N / 8, NW = RL_NT / 32;
  static_assert(M % 16 == 0 && N % 8 == 0, "MmaTile: M % 16 and N % 8");
  static_assert((MT * NT) % NW == 0, "MmaTile: tiles must divide over the warps");
  static constexpr int TPW = MT * NT / NW;
  static constexpr int CT = (NT < TPW) ? NT : TPW;
  static constexpr int RT = TPW / CT;
  static_assert(TPW % CT == 0 && NT % CT == 0 && MT % RT == 0, "MmaTile: warp tiling");
  static constexpr int WN = NT / CT;
  float acc[RT][CT][4];
  int row0, col0;

  __device__ __forceinline__ void init() {
    const int warp = threadIdx.x >> 5;
    row0 = (warp / WN) * RT * 16;
    col0 = (warp % WN) * CT * 8;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[r][c][e] = 0.f;
  }

  // acc += A[:, 0:K] * B[0:K, :]   (K % 8 == 0; A and B point at k = 0 of the chunk)
  // TF32: one MMA per fragment pair on rounded operands (inference precision RL_F_TF32) instead of the 3-pass split
  template <int AL, int BL, bool TF32 = false>
  __device__ __forceinline__ void mac(const float* __restrict__ A, int lda, const float* __restrict__ B, int ldb,
                                      int K) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll 2
    for (int k0 = 0; k0 < K; k0 += 8) {
      uint32_t ahi[RT][4], alo[RT][4];
#pragma unroll
      for (int r = 0; r < RT; ++r) {
        const int m = row0 + r * 16 + g;
        float a0, a1, a2, a3;
        if (AL == A_MK) {
          const float* p = A + m * lda + k0 + t;
          a0 = p[0]; a1 = p[8 * lda]; a2 = p[4]; a3 = p[8 * lda + 4];
        } else {
          const float* p = A + (k0 + t) * lda + m;
          a0 = p[0]; a1 = p[8]; a2 = p[4 * lda]; a3 = p[4 * lda + 8];
        }
        if constexpr (TF32) {
          ahi[r][0] = rna_tf32(a0); ahi[r][1] = rna_tf32(a1); ahi[r][2] = rna_tf32(a2); ahi[r][3] = rna_tf32(a3);
        } else {
          split_tf32x2(a0, a1, ahi[r][0], ahi[r][1], alo[r][0], alo[r][1]);
          split_tf32x2(a2, a3, ahi[r][2], ahi[r][3], alo[r][2], alo[r][3]);
        }
      }
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int n = col0 + c * 8 + g;
        float b0, b1;
        if (BL == B_NK) {
          const float* p = B + n * ldb + k0 + t;
          b0 = p[0]; b1 = p[4];
        } else {
          const float* p = B + (k0 + t) * ldb + n;
          b0 = p[0]; b1 = p[4 * ldb];
        }
        uint32_t bhi[2], blo[2];
        if constexpr (TF32) {
          bhi[0] = rna_tf32(b0); bhi[1] = rna_tf32(b1);
        } else {
          split_tf32x2(b0, b1, bhi[0], bhi[1], blo[0], blo[1]);
        }
#pragma unroll
        for (int r = 0; r < RT; ++r) {
          if constexpr (!TF32) {
            mma_tf32(acc[r][c], alo[r], bhi);
            mma_tf32(acc[r][c], ahi[r], blo);
          }
          mma_tf32(acc[r][c], ahi[r], bhi);
        }
      }
    }
  }

  // v[r][c][e] <- src[row * ld + col] for every output element owned by this thread, in the order of epilogue2():
  // all loads are issued back to back (one round trip to L2 / HBM instead of one per element inside an epilogue
  // lambda).  ld and the tile origin must be even (two adjacent columns per 8-byte load).
  // CG = true: the source was written earlier by THIS kernel (fused block kernels): L2-coherent loads instead of the
  // read-only path
  template <bool CG = false>
  __device__ __forceinline__ void gather(const float* src, int ld, float (&v)[RT][CT][4]) const {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int m = row0 + r * 16 + g, n = col0 + c * 8 + 2 * t;
        const float2* plo = reinterpret_cast<const float2*>(src + (size_t)m * ld + n);
        const float2* phi = reinterpret_cast<const float2*>(src + (size_t)(m + 8) * ld + n);
        const float2 lo = CG ? __ldcg(plo) : __ldg(plo);
        const float2 hi = CG ? __ldcg(phi) : __ldg(phi);
        v[r][c][0] = lo.x; v[r][c][1] = lo.y; v[r][c][2] = hi.x; v[r][c][3] = hi.y;
      }
  }
  // f(row, col, value, gathered value) for every output element owned by this thread
  template <class F>
  __device__ __forceinline__ void epilogue2(const float (&v)[RT][CT][4], F f) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int m = row0 + r * 16 + g, n = col0 + c * 8 + 2 * t;
        f(m, n, acc[r][c][0], v[r][c][0]);
        f(m, n + 1, acc[r][c][1], v[r][c][1]);
        f(m + 8, n, acc[r][c][2], v[r][c][2]);
        f(m + 8, n + 1, acc[r][c][3], v[r][c][3]);
      }
  }

  // pairs of adjacent columns: f(row, col, v0, v1) resp. f(row, col, v0, v1, gathered0, gathered1); col is even
  template <class F>
  __device__ __forceinline__ void epilogue_pairs(F f) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int m = row0 + r * 16 + g, n = col0 + c * 8 + 2 * t;
        f(m, n, acc[r][c][0], acc[r][c][1]);
        f(m + 8, n, acc[r][c][2], acc[r][c][3]);
      }
  }
  template <class F>
  __device__ __forceinline__ void epilogue2_pairs(const float (&v)[RT][CT][4], F f) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int m = row0 + r * 16 + g, n = col0 + c * 8 + 2 * t;
        f(m, n, acc[r][c][0], acc[r][c][1], v[r][c][0], v[r][c][1]);
        f(m + 8, n, acc[r][c][2], acc[r][c][3], v[r][c][2], v[r][c][3]);
      }
  }

  // f(row, col, value) for every output element owned by this thread
  template <class F>
  __device__ __forceinline__ void epilogue(F f) {
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const int m = row0 + r * 16 + g, n = col0 + c * 8 + 2 * t;
        f(m, n, acc[r][c][0]);
        f(m, n + 1, acc[r][c][1]);
        f(m + 8, n, acc[r][c][2]);
        f(m + 8, n + 1, acc[r][c][3]);
      }
  }
};

// shared-memory row strides that make the fragment loads of MmaTile conflict-free
__host__ __device__ constexpr int ld_mk(int K) { return K + 4; }                        // A_MK / B_NK: ld % 8 == 4
__host__ __device__ constexpr int ld_kn(int N) { return (N % 32 == 0) ? N + 8 : (N == 16 ? 24 : 40); }   // A_KM / B_KN
// largest power-of-two K chunk (>= 8) such that rows*(chunk+4) (B_NK) fits `budget` floats
__host__ __device__ constexpr int kc_nk(int N, int K, int budget) {
  int kc = K;
  while (kc > 8 && N * (kc + 4) > budget) kc /= 2;
  return kc;
}
// largest power-of-two K chunk (>= 8) such that chunk*ld_kn(N) (B_KN) fits `budget` floats
__host__ __device__ constexpr int kc_kn(int N, int K, int budget) {
  int kc = K;
  while (kc > 8 && kc * ld_kn(N) > budget) kc /= 2;
  return kc;
}
__host__ __device__ constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int SW_BUDGET = 6144;    // floats of weight staging per CTA at most (24 KB)

// copy `rows` rows of `cols` floats (cols % 4 == 0) from a dense global block to padded smem rows (float4)
__device__ __forceinline__ void copy_rows_g2s(float* dst, int ldd, const float* __restrict__ src, int rows, int cols) {
  const int c4n = cols >> 2;
  for (int i = threadIdx.x; i < rows * c4n; i += RL_NT) {
    const int r = i / c4n, c4 = i % c4n;
    *reinterpret_cast<float4*>(dst + r * ldd + 4 * c4) = __ldg(reinterpret_cast<const float4*>(src + r * cols) + c4);
  }
}
__device__ __forceinline__ void copy_rows_s2g(float* __restrict__ dst, const float* src, int lds, int rows, int cols) {
  const int c4n = cols >> 2;
  for (int i = threadIdx.x; i < rows * c4n; i += RL_NT) {
    const int r = i / c4n, c4 = i % c4n;
    reinterpret_cast<float4*>(dst + r * cols)[c4] = *reinterpret_cast<const float4*>(src + r * lds + 4 * c4);
  }
}

// ---------------------------------------------------------------------------------------------
// Weight streaming for the fused block kernels: the weight matrix stays in global memory (L2-resident, 4.3 MB
// for the whole network) and is pulled through a 2-stage cp.async ring in K chunks while the previous chunk is
// being contracted on the tensor cores.
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async16_zfill(float* smem_dst, const float* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int nbytes = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(nbytes));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int NPEND>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(NPEND)); }

constexpr int STAGE_BUDGET = 6144;   // floats per pipeline stage (24 KB)

// NS-stage ring of K chunks; BUDGET = floats per stage.  One __syncthreads per chunk: after the barrier of
// iteration c every thread has finished the MMAs of chunk c-1, so its stage is refilled with chunk c+NS-1.
// The first chunk can be issued long before the GEMM (prefetch(): before griddepcontrol.wait -- weights are never
// written by a kernel that triggers its dependents early -- or right after the previous GEMM on the same staging
// area), which hides the L2 latency of the weights behind the phase in between.
template <int N, int K, int BL, int NS = 2, int BUDGET = STAGE_BUDGET, int KSEG = K>
struct WStream {
  // KSEG: a chunk never straddles a multiple of KSEG (K = several concatenated operands of KSEG columns each)
  static constexpr int KC = (BL == B_NK) ? kc_nk(N, KSEG, BUDGET) : kc_kn(N, KSEG, BUDGET);
  static constexpr int LD = (BL == B_NK) ? KC + 4 : ld_kn(N);
  static constexpr int STAGE = (BL == B_NK) ? N * LD : KC * LD;     // floats per stage
  static constexpr int NCHUNK = K / KC;
  static constexpr int NSE = (NS < NCHUNK) ? NS : (NCHUNK < 2 ? 1 : NCHUNK);   // stages actually used
  static constexpr int FLOATS = NSE * STAGE;
  static_assert(K % KC == 0 && KC % 8 == 0 && NS >= 2, "WStream: chunking");

  // B_NK: W(n, k) = (n < split ? W0[n*ldw + k] : W1[(n-split)*ldw + k])         (y = x W^T, W = [N][K])
  // B_KN: W(k, n) = (k < split ? W0[k*ldw + n] : W1[(k-split)*ldw + n])         (dx = dy W,  W = [K][N])
  __device__ static __forceinline__ void issue(float* dst, const float* __restrict__ W0, int split,
                                               const float* __restrict__ W1, int ldw, int k0) {
    if (BL == B_NK) {
      constexpr int V = KC / 4;
      for (int i = threadIdx.x; i < N * V; i += RL_NT) {
        const int n = i / V, c = (i % V) * 4;
        const float* row = (n < split) ? W0 + (size_t)n * ldw : W1 + (size_t)(n - split) * ldw;
        cp_async16(dst + n * LD + c, row + k0 + c);
      }
    } else {
      constexpr int V = N / 4;
      for (int i = threadIdx.x; i < KC * V; i += RL_NT) {
        const int r = i / V, c = (i % V) * 4, k = k0 + r;
        const float* row = (k < split) ? W0 + (size_t)k * ldw : W1 + (size_t)(k - split) * ldw;
        cp_async16(dst + r * LD + c, row + c);
      }
    }
    cp_async_commit();
  }

  // issue chunk 0 into stage 0; the staging area must be free (a barrier since its last reader) and no other
  // cp.async group may be committed between this call and the matching run<true>()
  __device__ static __forceinline__ void prefetch(float* sw, const float* __restrict__ W0, int split,
                                                  const float* __restrict__ W1, int ldw) {
    issue(sw, W0, split, W1, ldw, 0);
  }

  // acc += A[:, 0:K] * W      (A in smem, A_MK with stride lda; sw holds FLOATS floats).  When the K range is the
  // concatenation of several A arrays (a_seg columns each, a_seg % KC == 0) the next one starts a_seg_stride floats
  // after the previous.  Ends with a barrier: afterwards sw (and A) may be overwritten.  TF32: see MmaTile::mac.
  template <bool PREFETCHED = false, bool TF32 = false, class Acc>
  __device__ static __forceinline__ void run(Acc& acc, const float* A, int lda, float* sw,
                                             const float* __restrict__ W0, int split,
                                             const float* __restrict__ W1, int ldw, int a_seg = K,
                                             int a_seg_stride = 0) {
    if (!PREFETCHED) issue(sw, W0, split, W1, ldw, 0);
#pragma unroll
    for (int s = 1; s < NSE - 1; ++s) issue(sw + s * STAGE, W0, split, W1, ldw, s * KC);
#pragma unroll 1
    for (int c = 0; c < NCHUNK; ++c) {
      cp_async_wait<(NSE >= 2) ? NSE - 2 : 0>();     // chunk c has landed (NSE-2 younger groups may be in flight)
      __syncthreads();
      if (NSE >= 2) {
        if (c + NSE - 1 < NCHUNK)
          issue(sw + ((c + NSE - 1) % NSE) * STAGE, W0, split, W1, ldw, (c + NSE - 1) * KC);
        else
          cp_async_commit();                          // empty group keeps the wait count static
      }
      const int k0 = c * KC;
      acc.template mac<A_MK, BL, TF32>(A + (k0 / a_seg) * a_seg_stride + (k0 % a_seg), lda, sw + (c % NSE) * STAGE, LD,
                                       KC);
    }
    __syncthreads();
  }
};

// ---------------------------------------------------------------------------------------------
// In-CTA weight gradient for the narrow stages (C <= 16), where a separate GEMM launch costs more than the math:
//   dW[n*K + k] += sum_{t<L} A[t*lda + n] * B[t*ldb + k]      db[n] += sum_t A[t*lda + n]
// on the tensor cores, in two phases around ONE CTA barrier:
//   partial(): every warp owns one (m16n8 tile of dW, token range) item -- rows = output features (padded to 16),
//     columns = input features, the L tokens split KS ways so that all 16 warps work (round 2 gave each tile to one warp
//     for all L tokens: at C = 16 two warps ran the MMAs while fourteen sat at the next barrier, 15 % of the samples of
//     attn_bwd<16> and 13 % of ffn_bwd<16> in ncu r2_v32) -- contracts it with 3xTF32 MMAs
//     (A(m = n_out, k = token) = A[t*lda + n], B(k = token, n = k_in) = B[t*ldb + k]) and leaves its fragment in
//     `scratch`; the warps of the first column tile also sum their A fragments over the tokens: the bias gradient.
//   reduce(): (after the barrier) adds the KS fragments of every element and issues one red.global per element of dW /
//     db and CTA (DET: one store into the CTA's slab slot).  No shared-memory atomics anywhere.
// Several partial()s into different scratch regions can share the barrier.
template <int N, int K, int L>
struct CtaWgrad {
  static_assert(K % 8 == 0, "CtaWgrad: K must be a multiple of 8");
  static constexpr int MT = (N + 15) / 16, NT = K / 8, NW = RL_NT / 32, TILES = MT * NT;
  static_assert(TILES <= NW && NW % TILES == 0, "CtaWgrad: the tiles must divide the warps");
  static constexpr int KS = NW / TILES, TOK = L / KS;
  static_assert(L % KS == 0 && TOK % 8 == 0, "CtaWgrad: token ranges must be multiples of 8");
  static constexpr int ITEM = 144;                       // floats per item: 32 lanes x 4 + 16 column sums
  static constexpr int SCRATCH = NW * ITEM;              // floats of scratch per call

  __device__ static __forceinline__ void partial(const float* A, int lda, const float* B, int ldb, float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, g = lane >> 2, t = lane & 3;
    const int tile = warp % TILES, ks = warp / TILES;
    const int m0 = (tile / NT) * 16, n0 = (tile % NT) * 8;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    float s_lo = 0.f, s_hi = 0.f;
    // rows >= N of a padded tile read the neighbouring smem words (in bounds) and are never stored
    const float* ap = A + (ks * TOK + t) * lda + m0 + g;
    const float* bp = B + (ks * TOK + t) * ldb + n0 + g;
#pragma unroll 4
    for (int k0 = 0; k0 < TOK; k0 += 8) {
      const float a0 = ap[k0 * lda], a1 = ap[k0 * lda + 8], a2 = ap[(k0 + 4) * lda], a3 = ap[(k0 + 4) * lda + 8];
      uint32_t ahi[4], alo[4], bhi[2], blo[2];
      split_tf32x2(a0, a1, ahi[0], ahi[1], alo[0], alo[1]);
      split_tf32x2(a2, a3, ahi[2], ahi[3], alo[2], alo[3]);
      split_tf32x2(bp[k0 * ldb], bp[(k0 + 4) * ldb], bhi[0], bhi[1], blo[0], blo[1]);
      mma_tf32(acc, alo, bhi);
      mma_tf32(acc, ahi, blo);
      mma_tf32(acc, ahi, bhi);
      if (n0 == 0) { s_lo += a0 + a2; s_hi += a1 + a3; }
    }
    float* item = scratch + warp * ITEM;                   // warp = ks * TILES + tile
    *reinterpret_cast<float4*>(item + 4 * lane) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    if (n0 == 0) {                                          // warp-uniform
      s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 1);
      s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 2);
      s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 1);
      s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 2);
      if (t == 0) { item[128 + g] = s_lo; item[136 + g] = s_hi; }
    }
  }

  template <bool DET = false>
  __device__ static __forceinline__ void reduce(const float* scratch, float* __restrict__ dW, float* __restrict__ db) {
    if (dW != nullptr) {
      for (int e = threadIdx.x; e < TILES * 128; e += RL_NT) {
        const int tile = e >> 7, idx = e & 127, ln = idx >> 2, j = idx & 3;
        float s = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) s += scratch[(ks * TILES + tile) * ITEM + idx];
        const int m = (tile / NT) * 16 + (ln >> 2) + ((j & 2) ? 8 : 0), n = (tile % NT) * 8 + 2 * (ln & 3) + (j & 1);
        if (m < N) grad_add<DET>(dW + m * K + n, s);
      }
    }
    if (db != nullptr) {
      for (int m = threadIdx.x; m < N; m += RL_NT) {
        const int tile = (m / 16) * NT;                     // the first column tile of this row block
        float s = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) s += scratch[(ks * TILES + tile) * ITEM + 128 + (m % 16)];
        grad_add<DET>(db + m, s);
      }
    }
  }
};

// true when every pointer is NULL or 16-byte aligned (the kernels use 16-byte accesses on activations, weights,
// LayerNorm vectors and the positional tile)
template <class... P>
inline bool rl_al16(P... p) { return (((uintptr_t)p | ...) & 15) == 0; }

// generic weight-gradient GEMM launcher (wgrad.cu):
//   dW[n*K + k] += sum_m dY[m*ldy + n] * X[m*ldx + k]      n < N, k < K, m < M
//   db[n]       += sum_m dY[m*ldy + n]                     (db may be NULL)
struct RlDet;
int rl_launch_wgrad(const float* dY, int ldy, const float* X, int ldx, int M, int N, int K, float* dW, float* db,
                    cudaStream_t st, RlDet* det = nullptr);
// grouped form: all weight matrices of one half-block in one launch (tensor-core path when every dim % 32 == 0)
struct RlWgradDesc {
  const float* dY; int ldy; const float* X; int ldx; int N, K; float* dW; float* db;
};
int rl_launch_wgrad_group(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det = nullptr);

// Deterministic-mode bookkeeping of one backward kernel and its weight-gradient GEMMs (net.cu): the partial slabs
// are carved from `slab` (cap floats) and every slab is recorded with the gradient it stands in for.
constexpr int RL_DET_MAXRED = 16;
constexpr int RL_DET_MAX_SPLIT = 148;   // token slices of a weight-gradient GEMM at most (bounds the slab size)
struct RlGradRed {
  const float* src;   // [slots][n]
  float* dst;         // [n] += sum over the slots, in slot order
  int n, slots;
};
struct RlDet {
  float* slab;
  size_t cap, used;
  RlGradRed red[RL_DET_MAXRED];
  int nred;
};
// slab region of slots x n floats standing in for gradient g (nullptr when g is nullptr or on overflow, with an error
// set: check rl_det_ok()); slab regions are 16-byte aligned
float* rl_det_take(RlDet* d, float* g, size_t n, int slots);
bool rl_det_ok(const RlDet* d);
// dst += sum over slots for every recorded slab, in one launch; clears the record
int rl_launch_grad_reduce(RlDet* d, cudaStream_t st);

// backward halves split into the data-gradient kernel and the weight-gradient GEMMs (net.cu runs the latter on a
// side stream, off the critical path of the backward chain).  det != nullptr: deterministic mode, the parameter
// gradients go to partial slabs recorded in *det (main and wgrad of one kernel share it)
int rl_attn_bwd_main(const rl_attn_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
int rl_attn_bwd_wgrad(const rl_attn_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
bool rl_attn_bwd_has_wgrad(const rl_attn_bwd_args* a);
int rl_ffn_bwd_main(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
int rl_ffn_bwd_wgrad(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
bool rl_ffn_bwd_has_wgrad(const rl_ffn_bwd_args* a);
int rl_patch_bwd_main(const rl_patch_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
int rl_patch_bwd_wgrad(const rl_patch_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
bool rl_patch_bwd_has_wgrad(const rl_patch_bwd_args* a);
int rl_head_bwd(const rl_head_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
int rl_stem_bwd_apply(const rl_stem_bwd_args* a, cudaStream_t st, RlDet* det = nullptr);
bool rl_prof_active();                 // per-launch profiling is on: keep every launch on the profiled stream
