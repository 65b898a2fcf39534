// attn.cu -- attention half of the RA-LENet TransformerBlock, one CTA per ECG window.
//
//   y = x + proj( softmax(0.5 q k^T + rw_bias) v ),   [q | k | v] = LN1(x*sqrt(C) + P) [Wq ; Wkv]^T + b
//
// Reference: model/transformer.py:383-390 (forward_part1), :289-323 (MSAttention), :226-247
// (LinearProjection), :179-181 (AbsPositionalEncoding), :534-558 (R-wave relative bias + mask_fill).
//
// A window is L tokens x C channels with L*C = 2048 (4096 for 512-sample windows), head_dim 4, so the
// whole window (x, q, k, v) lives in shared memory and the L x L logits are never materialised:
// each warp owns (head, 16-query tile) items and streams the keys through tensor-core MMAs with an online softmax
// (attn_core.cuh).  The R-wave bias is added from its (2W-1) x H table on the central W x W block only.
#define RL_NT 512        // 16 warps per window: the benchmark batch (256 windows on 148 SMs) needs the parallelism
#define RL_MINB 2
#include "common.cuh"
#include "attn_core.cuh"
#include "ffn_body.cuh"

RL_TRACE_DEFINE(attn)

int rl_attn_fwd_umma(const rl_attn_fwd_args* a, cudaStream_t st);       // tcgen05 tile kernels (attn_umma.cu)

namespace {

// weight streams: the wide stages pull their weights through deeper rings of smaller chunks (more loads in flight;
// a 2-stage ring leaves the L2 latency of every chunk exposed), sized so that two CTAs still fit on an SM
template <int C, int NS = ((C >= 64) ? 4 : 2)>
struct AttnW {
  using Qkv = WStream<3 * C, C, B_NK, NS, STAGE_BUDGET>;
  using Proj = WStream<C, C, B_NK, NS, (C >= 128) ? STAGE_BUDGET / 2 : STAGE_BUDGET>;
  using Dgrad = WStream<C, 3 * C, B_KN, NS, (C >= 64) ? STAGE_BUDGET / 2 : STAGE_BUDGET, C>;   // du = [dq|dk|dv] [Wq;Wkv]
  using DProj = WStream<C, C, B_KN, NS, (C >= 64) ? STAGE_BUDGET / 2 : STAGE_BUDGET>;          // do = g Wp
};
// forward: NWC windows per CTA.  At the wide stages a window has only 32 / 16 tokens while its CTA streams 64 / 256 KB
// of weights, and the kernel is bound by that L2 -> SM traffic (profiles/r1_v7_trace_attn.txt); two consecutive
// windows per CTA (M = 2L rows) halve it.  The 2-window variant keeps a 2-stage ring so that two CTAs still fit an SM.
template <int C, int NWC>
using AttnWF = AttnW<C, (NWC == 2) ? 2 : ((C >= 64) ? 4 : 2)>;
template <int C, int NWC>
__host__ __device__ constexpr int attn_fwd_swf() {
  return cmax(AttnWF<C, NWC>::Qkv::FLOATS, AttnWF<C, NWC>::Proj::FLOATS);
}
template <int C, int NWC>
size_t attn_fwd_smem(int L) {
  return sizeof(float) * (4 * (size_t)NWC * L * ld_mk(C) + attn_fwd_swf<C, NWC>() + 128);
}

// ---------------------------------------------------------------------------------------------
// TF32: single-pass projection GEMMs (RL_F_TF32, see MmaTile::mac); the attention core is the same in both forms
template <int C, int WIN, int NWC, bool TF32>
__device__ __forceinline__ void attn_fwd_body(const rl_attn_fwd_args& a, float* smem) {
  constexpr int L = 2048 * WIN / C, H = C / RL_HD, M = NWC * L;      // M token rows (NWC whole windows) per CTA
  constexpr int LDC = ld_mk(C);
  using WS = AttnWF<C, NWC>;
  const int W = a.W, c0 = a.c0;
  float* su = smem;
  float* sq = su + M * LDC;
  float* sk = sq + M * LDC;
  float* sv = sk + M * LDC;
  float* sw = sv + M * LDC;
  float* stab = sw + attn_fwd_swf<C, NWC>();
  // the weights are not produced by the preceding kernels of the step: start pulling them before the dependency wait
  RL_TS(attn, 0);
  WS::Qkv::prefetch(sw, a.wq, C, a.wkv, C);
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  RL_TS(attn, 1);
  const int tid = threadIdx.x;
  const size_t woff = (size_t)blockIdx.x * M * C;
  const float* xw = a.x + woff;

  // 1. x*sqrt(C) + P -> LayerNorm -> su          (transformer.py:386-387)
  if (a.flags & RL_F_PRENORM) {
    const float sc = sqrtf((float)C);
    const float* pe = a.pe;
    const float* lw = a.ln_w;
    const float* lb = a.ln_b;
    ln_forward_rows4<C>(
        M,
        [&](int t, int c) {
          const float4 x4 = ldg4(xw + t * C + c), p4 = ldg4(pe + (t % L) * C + c);
          return make_float4(fmaf(x4.x, sc, p4.x), fmaf(x4.y, sc, p4.y), fmaf(x4.z, sc, p4.z), fmaf(x4.w, sc, p4.w));
        },
        [&](int t, int c, float4 zh) { *reinterpret_cast<float4*>(su + t * LDC + c) = fma4(zh, ldg4(lw + c), ldg4(lb + c)); });
  } else {
    copy_rows_g2s(su, LDC, xw, M, C);
  }
  if (W > 0)
    for (int i = tid; i < (2 * W - 1) * H; i += RL_NT) stab[i] = __ldg(a.table + i) * RL_LOG2E;
  __syncthreads();
  RL_TS(attn, 2);

  // 2. [q|k|v] = u [Wq;Wkv]^T + b   (N = 3C, K = C): tensor-core GEMM, weights streamed through sw in K chunks
  {
    MmaTile<M, 3 * C> acc;
    acc.init();
    WS::Qkv::template run<true, TF32>(acc, su, LDC, sw, a.wq, C, a.wkv, C);
    WS::Proj::prefetch(sw, a.wp, C, nullptr, C);              // lands while the attention core runs
    const float* bq = a.bq;
    const float* bkv = a.bkv;
    acc.epilogue_pairs([&](int t, int n, float v0, float v1) {   // two adjacent columns: 8-byte bias loads and stores
      const int seg = n / C, c = n - seg * C;                    // q | k | v (a pair never straddles: C is even)
      const float* bsrc = (seg == 0) ? bq : bkv;
      if (bsrc) {
        const float2 b2 = __ldg(reinterpret_cast<const float2*>(bsrc + (seg == 2 ? C : 0) + c));
        v0 += b2.x;
        v1 += b2.y;
      }
      float* dst = (seg == 0) ? sq : (seg == 1) ? sk : sv;
      *reinterpret_cast<float2*>(dst + t * LDC + c) = make_float2(v0, v1);
    });
  }
  __syncthreads();
  RL_TS(attn, 3);
  if (a.q) {
    copy_rows_s2g(a.q + woff, sq, LDC, M, C);
    copy_rows_s2g(a.k + woff, sk, LDC, M, C);
    copy_rows_s2g(a.v + woff, sv, LDC, M, C);
  }
  RL_TS(attn, 4);

  // 3. attention core on the tensor cores (attn_core.cuh): one (head, 16-query tile) per warp, online softmax in
  //    the log2 domain; o overwrites q in place.  Windows attend only within themselves.
#pragma unroll
  for (int w = 0; w < NWC; ++w)
    attn_core_fwd<C, L>(sq + w * L * LDC, sk + w * L * LDC, sv + w * L * LDC, stab, W, c0,
                        a.lse ? a.lse + ((size_t)blockIdx.x * NWC + w) * H * L : nullptr);
  __syncthreads();
  RL_TS(attn, 5);
  if (a.o) copy_rows_s2g(a.o + woff, sq, LDC, M, C);
  RL_TS(attn, 6);

  // 4. y = x + o Wp^T + bp        (transformer.py:320, :405)
  {
    MmaTile<M, C> acc;
    acc.init();
    // residual: one batch of loads, issued BEFORE the projection GEMM so that their L2 round trip passes behind the
    // MMAs (ncu r2_v24: 8 % of the samples of block_fwd<16> sat on these loads when they followed the GEMM)
    float rv[MmaTile<M, C>::RT][MmaTile<M, C>::CT][4] = {};
    if (a.flags & RL_F_RESIDUAL) acc.gather(xw, C, rv);
    WS::Proj::template run<true, TF32>(acc, sq, LDC, sw, a.wp, C, nullptr, C);
    RL_TS(attn, 7);
    const float* bp = a.bp;
    float* yw = a.y + woff;
    acc.epilogue2_pairs(rv, [&](int t, int n, float v0, float v1, float add0, float add1) {
      if (bp) {
        const float2 b2 = __ldg(reinterpret_cast<const float2*>(bp + n));
        v0 += b2.x;
        v1 += b2.y;
      }
      *reinterpret_cast<float2*>(yw + t * C + n) = make_float2(v0 + add0, v1 + add1);
    });
  }
  RL_TS(attn, 8);
}

template <int C, int WIN, int NWC, bool TF32>
__global__ void __launch_bounds__(RL_NT, (NWC >= 4) ? 1 : RL_MINB) attn_fwd_kernel(const rl_attn_fwd_args a) {
  extern __shared__ __align__(16) float smem[];
  attn_fwd_body<C, WIN, NWC, TF32>(a, smem);
}

// One launch per TransformerBlock for the narrow stages (C <= 32, one window per CTA): attention half, then the
// feed-forward half on the block's own output.  x1 = f.x = a.y is written to global memory by the first half (the
// backward needs it anyway) and read back by the same CTA through L2-coherent loads after a CTA barrier; the second
// half's first weight chunk is requested before that barrier.  Saves a launch boundary (drain + fill + dependency
// wait) per block: 10 of the 36 block-half launches of a forward pass.
template <int C, bool TF32>
__global__ void __launch_bounds__(RL_NT, RL_MINB) block_fwd_kernel(const rl_attn_fwd_args a, const rl_ffn_fwd_args f) {
  extern __shared__ __align__(16) float smem[];
  attn_fwd_body<C, 1, 1, TF32>(a, smem);
  __syncthreads();                       // every thread's part of x1 is in global memory; the attention tiles are dead
  ffn_fwd_body<C, 1, true, TF32>(f, smem);
}

// ---------------------------------------------------------------------------------------------
template <int C>
__host__ __device__ constexpr int attn_bwd_swf() { return cmax(AttnW<C>::Dgrad::FLOATS, AttnW<C>::DProj::FLOATS); }
template <int C>
size_t attn_bwd_smem(int L) {
  return sizeof(float) * (8 * (size_t)L * ld_mk(C) + 2 * ((size_t)L * C / 4) + attn_bwd_swf<C>() + 256 + 2 * C);
}

template <int C, int WIN, bool DET>
__global__ void __launch_bounds__(RL_NT, RL_MINB) attn_bwd_kernel(const rl_attn_bwd_args a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int L = 2048 * WIN / C, H = C / RL_HD;
  constexpr int LDC = ld_mk(C), LC = L * C, LP = L * LDC;
  const int W = a.W, c0 = a.c0;
  float* sq = smem;
  float* sk = sq + LP;
  float* sv = sk + LP;
  float* sdo = sv + LP;
  float* sdq = sdo + LP;
  float* sdk = sdq + LP;
  float* sdv = sdk + LP;
  float* su = sdv + LP;
  float* sD = su + LP;
  float* sLse = sD + LC / 4;
  float* sw = sLse + LC / 4;
  float* stab = sw + attn_bwd_swf<C>();
  const int tid = threadIdx.x;
  __shared__ float s_amax[RL_NT / 32];
  RL_TS(attn, 0);
  const size_t woff = (size_t)blockIdx.x * LC;
  {   // The tensors the forward pass saved for this window -- q, k, v, o, lse -- do not depend on the preceding kernel
      // of the backward chain: they stream into shared memory with cp.async BEFORE the dependency wait (round 1 only
      // prefetched them to L2 and copied them after the wait: 10 % of the samples of attn_bwd<16> sat on those loads).
      // Their group is committed before the weight prefetch, so every later wait on a weight chunk covers it.
    constexpr int C4 = C / 4;
    for (int i = tid; i < L * C4; i += RL_NT) {
      const int r = i / C4, c = (i % C4) * 4;
      cp_async16(sq + r * LDC + c, a.q + woff + r * C + c);
      cp_async16(sk + r * LDC + c, a.k + woff + r * C + c);
      cp_async16(sv + r * LDC + c, a.v + woff + r * C + c);
      cp_async16(sdk + r * LDC + c, a.o + woff + r * C + c);
    }
    for (int i = tid; i < LC / 16; i += RL_NT) cp_async16(sLse + 4 * i, a.lse + (size_t)blockIdx.x * (LC / 4) + 4 * i);
    cp_async_commit();
    prefetch_l2_block(a.x + woff, LC * 4);                   // block input: needed by the LayerNorm backward at the end
  }
  AttnW<C>::DProj::prefetch(sw, a.wp, 1 << 30, nullptr, C);   // weights do not depend on the preceding kernels either
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  RL_TS(attn, 1);
  const float* gw = a.g + woff;
  const float* xw = a.x + woff;

  // 1. g -> sdq (temp); o sits in sdk (temp)
  copy_rows_g2s(sdq, LDC, gw, L, C);
  cp_async_wait<0>();                                        // saved tensors (and the first weight chunk) have landed
  for (int i = tid; i < LC / 16; i += RL_NT) {               // the core wants -lse: each thread negates the 16 bytes its
    float4* p = reinterpret_cast<float4*>(sLse + 4 * i);     // own cp.async wrote (visible to it after the wait above)
    const float4 v = *p;
    *p = make_float4(-v.x, -v.y, -v.z, -v.w);
  }
  if (tid < 128) {
    stab[tid] = (W > 0 && tid < (2 * W - 1) * H) ? __ldg(a.table + tid) * RL_LOG2E : 0.f;
  }
  __syncthreads();
  RL_TS(attn, 2);

  // 2. do = g Wp            (dgrad of proj; B(k,n) = Wp[k][n], natural layout)
  {
    MmaTile<L, C> acc;
    acc.init();
    AttnW<C>::DProj::template run<true>(acc, sdq, LDC, sw, a.wp, 1 << 30, nullptr, C);
    AttnW<C>::Dgrad::prefetch(sw, a.wq, C, a.wkv, C);         // lands while the attention core runs
    // max |do| of the window is taken from the accumulators on their way to shared memory (one barrier and one pass
    // over the tile less than reading it back)
    float am = 0.f;
    acc.epilogue_pairs([&](int t, int n, float v0, float v1) {
      *reinterpret_cast<float2*>(sdo + t * LDC + n) = make_float2(v0, v1);
      am = fmaxf(am, fmaxf(fabsf(v0), fabsf(v1)));
    });
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) am = fmaxf(am, __shfl_xor_sync(0xffffffffu, am, o));
    if ((tid & 31) == 0) s_amax[tid >> 5] = am;
  }
  __syncthreads();
  RL_TS(attn, 3);
  // 3. per-window power-of-two scale that puts max|do| at 2^6 (the single-pass core carries its operands as fp16
  //    hi/lo pairs; gradients are ~1e-6 and would underflow unscaled), then D[h,i] = do_i . o_i (scaled alike)
  float do_scale;
  {
    float am = s_amax[0];
#pragma unroll
    for (int w = 1; w < RL_NT / 32; ++w) am = fmaxf(am, s_amax[w]);
    do_scale = (am > 0.f && am < 3e38f) ? exp2f(6.f - ceilf(log2f(am))) : 1.f;
  }
  for (int item = tid; item < H * L; item += RL_NT) {
    const int i = item % L, h = item / L;
    const float4 d4 = *reinterpret_cast<const float4*>(sdo + i * LDC + 4 * h);
    const float4 o4 = *reinterpret_cast<const float4*>(sdk + i * LDC + 4 * h);
    sD[item] = -do_scale * (d4.x * o4.x + d4.y * o4.y + d4.z * o4.z + d4.w * o4.w);     // the core wants -D
  }
  __syncthreads();

  constexpr bool FW = (C <= RL_FW_MAXC);   // narrow stages: weight gradients are accumulated in-CTA (no wgrad launch)
  if constexpr (FW) {                      // dWp = g^T o,  dbp = sum g; su is free until step 6
    static_assert(CtaWgrad<C, C, L>::SCRATCH <= LP, "attn_bwd: scratch");
    CtaWgrad<C, C, L>::partial(sdq, LDC, sdk, LDC, su);
    __syncthreads();
    CtaWgrad<C, C, L>::template reduce<DET>(su, grad_slot<DET>(a.d_wp, C * C, blockIdx.x),
                                            grad_slot<DET>(a.d_bp, C, blockIdx.x));
  }
  RL_TS(attn, 4);

  // 4. attention core backward on the tensor cores (attn_core.cuh), single pass: q, k, v, do are re-packed in place
  //    as fp16 hi/lo pairs, one warp per (head, 16-key tile) walks the queries once; p is recomputed from the saved
  //    log-sum-exp; dq partial sums meet in shared-memory reds (sdq held g, sdk held o: both dead by now).
  to_row_form<C>(sq, LDC, L, 0.5f * RL_LOG2E);
  to_row_form<C>(sk, LDC, L, 1.f);
  to_row_form<C>(sv, LDC, L, 1.f);
  to_row_form<C>(sdo, LDC, L, do_scale);
  for (int i = tid; i < LP; i += RL_NT) sdq[i] = 0.f;
  __syncthreads();
  RL_TS(attn, 5);
  float* sds_c = (a.d_table != nullptr && W > 0) ? su : nullptr;      // su is free until step 6 (H * W * W <= LP floats)
  attn_core_bwd_single<C, L>(sq, sk, sv, sdo, sD, sLse, sdq, sdk, sdv, stab, sds_c, W, c0, 1.0f / do_scale);
  __syncthreads();
  if (sds_c != nullptr) {         // d_table[i - j + W - 1][h] += sum over the diagonal of the central block of dS
    float* d_table = grad_slot<DET>(a.d_table, (2 * W - 1) * H, blockIdx.x);
    for (int idx = tid; idx < (2 * W - 1) * H; idx += RL_NT) {
      const int rel = idx / H - (W - 1), h = idx % H;
      const int jlo = (rel < 0) ? -rel : 0, jhi = (rel > 0) ? W - rel : W;
      float s = 0.f;
      for (int j = jlo; j < jhi; ++j) s += sds_c[(h * W + j + rel) * W + j];
      grad_add<DET>(d_table + idx, s);
    }
  }
  RL_TS(attn, 6);

  // 5. dqkv scratch [t][dq | dk | dv] for the weight-gradient GEMMs
  if (!FW) {
    float* dst = a.dqkv + (size_t)blockIdx.x * 3 * LC;
    constexpr int C4 = C / 4;
    for (int i = tid; i < 3 * L * C4; i += RL_NT) {
      const int c4 = i % C4, seg = (i / C4) % 3, t = i / (3 * C4);
      const float* src = (seg == 0) ? sdq : (seg == 1) ? sdk : sdv;
      reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(src + t * LDC)[c4];
    }
  }

  RL_TS(attn, 7);
  // 6. du = [dq | dk | dv] [Wq ; Wk ; Wv]      (K = 3C: one weight stream over the three row blocks; sdq, sdk, sdv
  //    are consecutive L x LDC arrays)
  {
    MmaTile<L, C> acc;
    acc.init();
    AttnW<C>::Dgrad::template run<true>(acc, sdq, LDC, sw, a.wq, C, a.wkv, C, C, LP);
    acc.epilogue_pairs([&](int t, int n, float v0, float v1) {
      *reinterpret_cast<float2*>(su + t * LDC + n) = make_float2(v0, v1);
    });
  }
  __syncthreads();

  RL_TS(attn, 8);
  // 7. LayerNorm backward, positional scale, residual
  float* dxw = a.dx + woff;
  float* uw = a.u + woff;
  const bool resid = a.flags & RL_F_RESIDUAL;
  if (a.flags & RL_F_PRENORM) {
    const float sc = sqrtf((float)C);
    const float* pe = a.pe;
    const float* lw = a.ln_w;
    const float* lb = a.ln_b;
    // per-warp partial rows of the LayerNorm weight / bias gradients go to sq..sk (16 x 2C floats; q, k are dead)
    ln_backward_rows4<C, true>(
        L, lw, sq,
        [&](int t, int c) {
          const float4 x4 = ldg4(xw + t * C + c), p4 = ldg4(pe + t * C + c);
          return make_float4(fmaf(x4.x, sc, p4.x), fmaf(x4.y, sc, p4.y), fmaf(x4.z, sc, p4.z), fmaf(x4.w, sc, p4.w));
        },
        [&](int t, int c) { return *reinterpret_cast<const float4*>(su + t * LDC + c); },
        [&](int t, int c, float4 dz, float4 zh) {
          const float4 g4 = resid ? ldg4(gw + t * C + c) : make_float4(0.f, 0.f, 0.f, 0.f);
          *reinterpret_cast<float4*>(dxw + t * C + c) =
              make_float4(fmaf(sc, dz.x, g4.x), fmaf(sc, dz.y, g4.y), fmaf(sc, dz.z, g4.z), fmaf(sc, dz.w, g4.w));
          const float4 u = fma4(zh, ldg4(lw + c), ldg4(lb + c));
          // du at (t, c..c+3) was consumed by this thread
          *reinterpret_cast<float4*>(FW ? su + t * LDC + c : uw + t * C + c) = u;
        });
    __syncthreads();
    ln_backward_finish<C, DET>(sq, grad_slot<DET>(a.d_ln_w, C, blockIdx.x), grad_slot<DET>(a.d_ln_b, C, blockIdx.x));
  } else {
    for (int i = tid; i < LC; i += RL_NT) {
      const int t = i / C, c = i % C;
      dxw[i] = su[t * LDC + c] + (resid ? __ldg(gw + i) : 0.f);
      if (FW) su[t * LDC + c] = __ldg(xw + i); else uw[i] = __ldg(xw + i);
    }
    __syncthreads();
  }
  RL_TS(attn, 9);
  if constexpr (FW) {   // dWq = dq^T u, dWkv = [dk | dv]^T u  (u now sits in su); scratch: sk, sv, sdo (dead since the core)
    using WG = CtaWgrad<C, C, L>;
    static_assert(WG::SCRATCH <= LP && 16 * 2 * C <= LP, "attn_bwd: scratch regions");
    WG::partial(sdq, LDC, su, LDC, sk);
    WG::partial(sdk, LDC, su, LDC, sv);
    WG::partial(sdv, LDC, su, LDC, sdo);
    __syncthreads();
    float* d_wkv = grad_slot<DET>(a.d_wkv, 2 * C * C, blockIdx.x);
    float* d_bkv = grad_slot<DET>(a.d_bkv, 2 * C, blockIdx.x);
    WG::template reduce<DET>(sk, grad_slot<DET>(a.d_wq, C * C, blockIdx.x), grad_slot<DET>(a.d_bq, C, blockIdx.x));
    WG::template reduce<DET>(sv, d_wkv, d_bkv);
    WG::template reduce<DET>(sdo, d_wkv ? d_wkv + C * C : nullptr, d_bkv ? d_bkv + C : nullptr);
  }
  RL_TS(attn, 10);
}

#ifndef RL_NWC_MIN_B
#define RL_NWC_MIN_B 512      // batches at least this large put two windows on a CTA at the wide stages (at the
#endif                        // benchmark batch of 256 the halved CTA count costs more than the weight traffic saves)
// (four windows per CTA at C = 128 -- one 170 KB CTA per SM -- measured slower than two: 320 vs 294 us at B = 4096)

// `a` advanced by w0 windows, n windows long
rl_attn_fwd_args attn_fwd_slice(const rl_attn_fwd_args& a, int w0, int n) {
  rl_attn_fwd_args s = a;
  const size_t off = (size_t)w0 * a.L * a.C;
  s.B = n;
  s.x = a.x + off;
  s.y = a.y + off;
  if (a.q) { s.q = a.q + off; s.k = a.k + off; s.v = a.v + off; s.o = a.o + off; }
  if (a.lse) s.lse = a.lse + (size_t)w0 * a.H * a.L;
  return s;
}

// launches floor(B / NWC) CTAs of NWC windows each; returns the number of windows covered through *done
template <int C, int NWC, bool TF32>
int launch_fwd_groups(const rl_attn_fwd_args* a, cudaStream_t st, int* done) {
  const size_t smem = attn_fwd_smem<C, NWC>(a->L);
  if (int rc = rl_set_smem(attn_fwd_kernel<C, 1, NWC, TF32>, smem)) return rc;
  rl_launch_pdl(attn_fwd_kernel<C, 1, NWC, TF32>, dim3(a->B / NWC), dim3(RL_NT), smem, st, *a);
  *done = (a->B / NWC) * NWC;
  return rl_check_launch("attn_fwd_kernel", C, NWC, rl_tf32_tag(TF32));
}

template <int C, bool TF32>
int launch_fwd(const rl_attn_fwd_args* a, cudaStream_t st) {
  const int win = a->L * C / 2048;
  if (win != 1) {
    const size_t smem = attn_fwd_smem<C, 1>(a->L);
    if (int rc = rl_set_smem(attn_fwd_kernel<C, 2, 1, TF32>, smem)) return rc;
    rl_launch_pdl(attn_fwd_kernel<C, 2, 1, TF32>, dim3(a->B), dim3(RL_NT), smem, st, *a);
    return rl_check_launch("attn_fwd_kernel", C, -1, rl_tf32_tag(TF32));
  }
  if (C >= 64) {
    const int rc = rl_attn_fwd_umma(a, st);                      // 1: shape / batch not handled there
    if (rc <= 0) return rc;
  }
  int done = 0;
  if (C >= 64 && a->B >= RL_NWC_MIN_B) {
    if (int rc = launch_fwd_groups<C, (C >= 64) ? 2 : 1, TF32>(a, st, &done)) return rc;
  }
  if (done == a->B) return RL_OK;
  const rl_attn_fwd_args rest = attn_fwd_slice(*a, done, a->B - done);     // the odd windows, one per CTA
  int d1 = 0;
  return launch_fwd_groups<C, 1, TF32>(&rest, st, &d1);
}
template <int C>
int launch_fwd(const rl_attn_fwd_args* a, cudaStream_t st) {
  return (a->flags & RL_F_TF32) ? launch_fwd<C, true>(a, st) : launch_fwd<C, false>(a, st);
}

template <int C, int WIN, bool DET>
int launch_bwd_one(const rl_attn_bwd_args* a, cudaStream_t st) {
  const size_t smem = attn_bwd_smem<C>(a->L);
  if (int rc = rl_set_smem(attn_bwd_kernel<C, WIN, DET>, smem)) return rc;
  rl_launch_pdl(attn_bwd_kernel<C, WIN, DET>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  return rl_check_launch("attn_bwd_kernel", C);
}

// det: one partial slot per window (CTA) for the in-CTA gradients (LayerNorm, R-wave table; every weight at C <= 16)
template <int C>
int launch_bwd(const rl_attn_bwd_args* a, cudaStream_t st, RlDet* det) {
  const int win = a->L * C / 2048;
  if (det == nullptr) return win == 1 ? launch_bwd_one<C, 1, false>(a, st) : launch_bwd_one<C, 2, false>(a, st);
  rl_attn_bwd_args d = *a;
  const int B = a->B;
  d.d_ln_w = rl_det_take(det, a->d_ln_w, C, B);
  d.d_ln_b = rl_det_take(det, a->d_ln_b, C, B);
  d.d_table = (a->W > 0) ? rl_det_take(det, a->d_table, (2 * a->W - 1) * (C / RL_HD), B) : nullptr;
  if (C <= RL_FW_MAXC) {
    d.d_wq = rl_det_take(det, a->d_wq, C * C, B);   d.d_bq = rl_det_take(det, a->d_bq, C, B);
    d.d_wkv = rl_det_take(det, a->d_wkv, 2 * C * C, B); d.d_bkv = rl_det_take(det, a->d_bkv, 2 * C, B);
    d.d_wp = rl_det_take(det, a->d_wp, C * C, B);   d.d_bp = rl_det_take(det, a->d_bp, C, B);
  }
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "attn_bwd: deterministic-mode workspace too small");
  return win == 1 ? launch_bwd_one<C, 1, true>(&d, st) : launch_bwd_one<C, 2, true>(&d, st);
}

int check_shape(int B, int L, int C, int H, int W, int c0) {
  RL_REQUIRE(B > 0, RL_ERR_SHAPE, "attn: B=%d", B);
  RL_REQUIRE(C == 8 || C == 16 || C == 32 || C == 64 || C == 128, RL_ERR_SHAPE, "attn: unsupported C=%d", C);
  RL_REQUIRE(H * RL_HD == C, RL_ERR_SHAPE, "attn: head_dim must be 4 (C=%d, H=%d)", C, H);
  RL_REQUIRE(L * C == 2048 || L * C == 4096, RL_ERR_SHAPE, "attn: L*C must be 2048 or 4096 (L=%d, C=%d)", L, C);
  RL_REQUIRE(W >= 0 && (W == 0 || (c0 >= 0 && c0 + W <= L && (2 * W - 1) * H <= 128)), RL_ERR_SHAPE,
             "attn: bad R-wave window W=%d c0=%d L=%d H=%d", W, c0, L, H);
  return RL_OK;
}

template <int C, bool TF32>
int launch_block_fwd(const rl_attn_fwd_args* a, const rl_ffn_fwd_args* f, cudaStream_t st) {
  const size_t s1 = attn_fwd_smem<C, 1>(a->L), s2 = ffn_fwd_smem<C>(a->L);
  const size_t smem = s1 > s2 ? s1 : s2;
  if (int rc = rl_set_smem(block_fwd_kernel<C, TF32>, smem)) return rc;
  rl_launch_pdl(block_fwd_kernel<C, TF32>, dim3(a->B), dim3(RL_NT), smem, st, *a, *f);
  return rl_check_launch("block_fwd_kernel", C, -1, rl_tf32_tag(TF32));
}
template <int C>
int launch_block_fwd(const rl_attn_fwd_args* a, const rl_ffn_fwd_args* f, cudaStream_t st) {
  return (a->flags & RL_F_TF32) ? launch_block_fwd<C, true>(a, f, st) : launch_block_fwd<C, false>(a, f, st);
}

int g_block_fuse = -1;
int block_fuse_on() {
  if (g_block_fuse < 0) {
    const char* e = getenv("RALENET_BLOCK_FUSE");
    g_block_fuse = (e && e[0] == '0') ? 0 : 1;
  }
  return g_block_fuse;
}

}  // namespace

extern "C" int ralenet_set_block_fuse(int on) {
  const int prev = block_fuse_on();
  g_block_fuse = on ? 1 : 0;
  return prev;
}

// TransformerBlock.forward (model/transformer.py:398-411) = attention half + feed-forward half.  Narrow stages
// (C <= 32, 256-sample windows, both halves pre-norm + residual, f->x == a->y): ONE fused launch; anything else: the
// two halves one after the other.
extern "C" int ralenet_block_fwd(const rl_attn_fwd_args* a, const rl_ffn_fwd_args* f, void* stream) {
  RL_REQUIRE(a && f, RL_ERR_NULL, "block_fwd: args is NULL");
  RL_REQUIRE(((a->flags ^ f->flags) & RL_F_TF32) == 0, RL_ERR_SHAPE, "block_fwd: the halves differ in RL_F_TF32");
  const int want = RL_F_PRENORM | RL_F_RESIDUAL;
  const bool fuse = block_fuse_on() && a->C <= 32 && a->L * a->C == 2048 && f->x == a->y && f->B == a->B &&
                    f->L == a->L && f->C == a->C && (a->flags & want) == want && (f->flags & want) == want &&
                    f->le_mode != RL_LE_DEPTHWISE;
  if (!fuse) {
    if (int rc = ralenet_attn_fwd(a, stream)) return rc;
    return ralenet_ffn_fwd(f, stream);
  }
  if (int rc = check_shape(a->B, a->L, a->C, a->H, a->W, a->c0)) return rc;
  RL_REQUIRE(a->x && a->y && a->wq && a->wkv && a->wp && a->pe && a->ln_w && a->ln_b, RL_ERR_NULL,
             "block_fwd: NULL attention tensor");
  RL_REQUIRE(a->W == 0 || a->table, RL_ERR_NULL, "block_fwd: W>0 needs table");
  RL_REQUIRE(!a->q || (a->k && a->v && a->o && a->lse), RL_ERR_NULL, "block_fwd: partial save set");
  RL_REQUIRE(!(a->flags & RL_F_TF32) || !(a->q || a->k || a->v || a->o || a->lse || f->h), RL_ERR_SHAPE,
             "block_fwd: RL_F_TF32 is inference only (saved-tensor pointers must be NULL)");
  RL_REQUIRE(f->y && f->w1 && f->w2 && f->ln_w && f->ln_b, RL_ERR_NULL, "block_fwd: NULL feed-forward tensor");
  RL_REQUIRE(f->le_mode == RL_LE_NONE || f->lew, RL_ERR_NULL, "block_fwd: local-enhancement weights missing");
  RL_REQUIRE(rl_al16(a->x, a->y, a->pe, a->ln_w, a->ln_b, a->wq, a->wkv, a->wp, a->q, a->k, a->v, a->o, f->y, f->w1, f->w2,
                     f->ln_w, f->ln_b, f->h, f->extra),
             RL_ERR_SHAPE, "block_fwd: tensors must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  switch (a->C) {
    case 8: return launch_block_fwd<8>(a, f, st);
    case 16: return launch_block_fwd<16>(a, f, st);
    case 32: return launch_block_fwd<32>(a, f, st);
  }
  return RL_ERR_SHAPE;
}

extern "C" int ralenet_attn_fwd(const rl_attn_fwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "attn_fwd: args is NULL");
  if (int rc = check_shape(a->B, a->L, a->C, a->H, a->W, a->c0)) return rc;
  RL_REQUIRE(a->x && a->y && a->wq && a->wkv && a->wp, RL_ERR_NULL, "attn_fwd: NULL tensor");
  RL_REQUIRE(!(a->flags & RL_F_PRENORM) || (a->pe && a->ln_w && a->ln_b), RL_ERR_NULL, "attn_fwd: prenorm needs pe/ln");
  RL_REQUIRE(a->W == 0 || a->table, RL_ERR_NULL, "attn_fwd: W>0 needs table");
  RL_REQUIRE(!a->q || (a->k && a->v && a->o && a->lse), RL_ERR_NULL, "attn_fwd: partial save set");
  RL_REQUIRE(!(a->flags & RL_F_TF32) || !(a->q || a->k || a->v || a->o || a->lse), RL_ERR_SHAPE,
             "attn_fwd: RL_F_TF32 is inference only (q/k/v/o/lse must be NULL)");
  RL_REQUIRE(rl_al16(a->x, a->y, a->pe, a->ln_w, a->ln_b, a->wq, a->wkv, a->wp, a->q, a->k, a->v, a->o), RL_ERR_SHAPE,
             "attn_fwd: tensors must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  switch (a->C) {
    case 8: return launch_fwd<8>(a, st);
    case 16: return launch_fwd<16>(a, st);
    case 32: return launch_fwd<32>(a, st);
    case 64: return launch_fwd<64>(a, st);
    case 128: return launch_fwd<128>(a, st);
  }
  return RL_ERR_SHAPE;
}

// the data-gradient kernel (also writes the dqkv / u scratch of the weight gradients)
int rl_attn_bwd_main(const rl_attn_bwd_args* a, cudaStream_t st, RlDet* det) {
  RL_REQUIRE(a, RL_ERR_NULL, "attn_bwd: args is NULL");
  RL_REQUIRE(!(a->flags & RL_F_TF32), RL_ERR_SHAPE, "attn_bwd: RL_F_TF32 is a forward-only (inference) flag");
  if (int rc = check_shape(a->B, a->L, a->C, a->H, a->W, a->c0)) return rc;
  RL_REQUIRE(a->g && a->x && a->wq && a->wkv && a->wp && a->q && a->k && a->v && a->o && a->lse && a->dx && a->dqkv &&
                 a->u,
             RL_ERR_NULL, "attn_bwd: NULL tensor");
  RL_REQUIRE(!(a->flags & RL_F_PRENORM) || (a->pe && a->ln_w && a->ln_b), RL_ERR_NULL, "attn_bwd: prenorm needs pe/ln");
  RL_REQUIRE(a->W == 0 || a->table, RL_ERR_NULL, "attn_bwd: W>0 needs table");
  RL_REQUIRE(!a->d_ln_w == !a->d_ln_b, RL_ERR_NULL, "attn_bwd: d_ln_w/d_ln_b must be both set or both NULL");
  RL_REQUIRE(rl_al16(a->g, a->x, a->pe, a->ln_w, a->ln_b, a->wq, a->wkv, a->wp, a->q, a->k, a->v, a->o, a->lse, a->dx,
                     a->dqkv, a->u),
             RL_ERR_SHAPE, "attn_bwd: tensors must be 16-byte aligned");
  switch (a->C) {
    case 8: return launch_bwd<8>(a, st, det);
    case 16: return launch_bwd<16>(a, st, det);
    case 32: return launch_bwd<32>(a, st, det);
    case 64: return launch_bwd<64>(a, st, det);
    case 128: return launch_bwd<128>(a, st, det);
  }
  return RL_ERR_SHAPE;
}

// true when the weight gradients of this shape are a separate launch (rl_attn_bwd_wgrad)
bool rl_attn_bwd_has_wgrad(const rl_attn_bwd_args* a) {
  return a->C > RL_FW_MAXC && (a->d_wp || a->d_wq || a->d_wkv);
}

// weight gradients from (g, o) and the scratch tensors; may run on another stream once the main kernel is done
int rl_attn_bwd_wgrad(const rl_attn_bwd_args* a, cudaStream_t st, RlDet* det) {
  const int M = a->B * a->L, C = a->C;
  if (C <= RL_FW_MAXC) return RL_OK;        // narrow stages accumulate their weight gradients inside the kernel
  const RlWgradDesc d[3] = {{a->g, C, a->o, C, C, C, a->d_wp, a->d_bp},
                            {a->dqkv, 3 * C, a->u, C, C, C, a->d_wq, a->d_bq},
                            {a->dqkv + C, 3 * C, a->u, C, 2 * C, C, a->d_wkv, a->d_bkv}};
  return rl_launch_wgrad_group(d, 3, M, st, det);
}

extern "C" int ralenet_attn_bwd(const rl_attn_bwd_args* a, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = rl_attn_bwd_main(a, st)) return rc;
  return rl_attn_bwd_wgrad(a, st);
}
