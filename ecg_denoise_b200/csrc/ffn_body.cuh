// ffn_body.cuh -- forward of the feed-forward half for one window per CTA as a device function, shared by
// ffn.cu (the stand-alone kernel) and attn.cu (second half of the fused block kernel of the narrow stages).
#pragma once
#include "common.cuh"

template <int C>
__host__ __device__ constexpr int ffn_fwd_swf() {
  return cmax(WStream<4 * C, C, B_NK>::FLOATS, WStream<C, 4 * C, B_NK>::FLOATS);
}
template <int C>
size_t ffn_fwd_smem(int L) {
  return sizeof(float) * ((size_t)L * ld_mk(C) + (size_t)L * ld_mk(4 * C) + ffn_fwd_swf<C>() + (size_t)L + 64);
}

// CHAIN = true: second half of a fused block kernel (attn.cu::block_fwd_kernel): the input a.x was written by this
// very CTA a moment ago (the attention half's output), so there is no programmatic-dependency wait and the input is
// read with L2-coherent loads.  TF32: single-pass GEMMs (RL_F_TF32, see MmaTile::mac).
template <int C, int WIN, bool CHAIN, bool TF32>
__device__ __forceinline__ void ffn_fwd_body(const rl_ffn_fwd_args& a, float* smem) {
  constexpr int L = 2048 * WIN / C;
  constexpr int LDC = ld_mk(C);
  constexpr int HC = 4 * C, LDH = ld_mk(HC);
  float* su = smem;
  float* sh = su + L * LDC;
  float* sw = sh + L * LDH;
  float* sfir = sw + ffn_fwd_swf<C>();
  // the weights are not produced by the preceding kernels of the step: start pulling them before the dependency wait
  WStream<HC, C, B_NK>::prefetch(sw, a.w1, HC, nullptr, C);
  if (!CHAIN) {
    pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
    pdl_trigger();   // let the next kernel get scheduled while this one runs
  }
  const int tid = threadIdx.x;
  const size_t woff = (size_t)blockIdx.x * L * C;
  const float* xw = a.x + woff;

  // 1. LN2
  if (a.flags & RL_F_PRENORM) {
    const float* lw = a.ln_w;
    const float* lb = a.ln_b;
    ln_forward_rows4<C>(
        L,
        [&](int t, int c) {
          const float4* p4 = reinterpret_cast<const float4*>(xw + t * C + c);
          return CHAIN ? __ldcg(p4) : __ldg(p4);
        },
        [&](int t, int c, float4 zh) { *reinterpret_cast<float4*>(su + t * LDC + c) = fma4(zh, ldg4(lw + c), ldg4(lb + c)); });
  } else {
    copy_rows_g2s(su, LDC, xw, L, C);
  }
  __syncthreads();

  // 2. h = u W1^T + b1 (N = 4C, K = C);  g1 = GELU(h) -> sh
  {
    MmaTile<L, HC> acc;
    acc.init();
    WStream<HC, C, B_NK>::template run<true, TF32>(acc, su, LDC, sw, a.w1, HC, nullptr, C);
    WStream<C, HC, B_NK>::prefetch(sw, a.w2, C, nullptr, HC);      // lands behind the GELU / local-enhancement phase
    const float* b1 = a.b1;
    float* hs = a.h ? a.h + (size_t)blockIdx.x * L * HC : nullptr;
    const bool partial = (a.le_mode == RL_LE_PARTIAL);
    acc.epilogue_pairs([&](int t, int n, float v0, float v1) {      // two hidden units per call: packed-fp32 GELU
      if (b1) { v0 += __ldg(b1 + n); v1 += __ldg(b1 + n + 1); }
      if (hs) *reinterpret_cast<float2*>(hs + t * HC + n) = make_float2(v0, v1);
      float g0, g1;
      gelu2(v0, v1, g0, g1);
      if (partial) {
        // partial local enhancement: only hidden unit 0 is convolved, every other unit goes straight through the
        // second GELU here, in registers (round 2 made a second pass over the whole L x 4C tile in shared memory)
        float q0, q1;
        gelu2(g0, g1, q0, q1);
        g1 = q1;
        if (n != 0) g0 = q0;                                        // unit 0 keeps GELU(h): FIR + GELU below
      }
      *reinterpret_cast<float2*>(sh + t * LDH + n) = make_float2(g0, g1);
    });
  }
  __syncthreads();

  // 3. local enhancement + second GELU
  if (a.le_mode == RL_LE_PARTIAL) {
    const float w0 = __ldg(a.lew), w1 = __ldg(a.lew + 1), w2 = __ldg(a.lew + 2);
    for (int t = tid; t < L; t += RL_NT) {
      const float p = (t > 0) ? sh[(t - 1) * LDH] : 0.f;
      const float n = (t + 1 < L) ? sh[(t + 1) * LDH] : 0.f;
      sfir[t] = w0 * p + w1 * sh[t * LDH] + w2 * n;
    }
    __syncthreads();
    for (int t = tid; t < L; t += RL_NT) sh[t * LDH] = gelu_f(sfir[t]);
    __syncthreads();
  } else if (a.le_mode == RL_LE_DEPTHWISE) {
    for (int c = tid; c < HC; c += RL_NT) {
      const float w0 = __ldg(a.lew + 3 * c), w1 = __ldg(a.lew + 3 * c + 1), w2 = __ldg(a.lew + 3 * c + 2);
      float prev = 0.f, cur = sh[c];
      for (int t = 0; t < L; ++t) {
        const float nxt = (t + 1 < L) ? sh[(t + 1) * LDH + c] : 0.f;
        sh[t * LDH + c] = gelu_f(w0 * prev + w1 * cur + w2 * nxt);
        prev = cur;
        cur = nxt;
      }
    }
    __syncthreads();
  }

  // 4. y = x + g2 W2^T + b2 (N = C, K = 4C)
  {
    MmaTile<L, C> acc;
    acc.init();
    const bool resid = a.flags & RL_F_RESIDUAL;
    // residual (and the U-net skip of the middle block): one batch of loads, not one round trip per element -- issued
    // before the fc2 GEMM so that the round trip passes behind the MMAs
    float rv[MmaTile<L, C>::RT][MmaTile<L, C>::CT][4] = {}, ev[MmaTile<L, C>::RT][MmaTile<L, C>::CT][4] = {};
    if (resid) acc.template gather<CHAIN>(xw, C, rv);
    WStream<C, HC, B_NK>::template run<true, TF32>(acc, sh, LDH, sw, a.w2, C, nullptr, HC);
    const float* b2 = a.b2;
    const float* ex = a.extra ? a.extra + woff : nullptr;
    float* yw = a.y + woff;
    if (ex) {
      acc.gather(ex, C, ev);
#pragma unroll
      for (int r = 0; r < MmaTile<L, C>::RT; ++r)
#pragma unroll
        for (int c = 0; c < MmaTile<L, C>::CT; ++c)
#pragma unroll
          for (int e = 0; e < 4; ++e) rv[r][c][e] += ev[r][c][e];
    }
    acc.epilogue2_pairs(rv, [&](int t, int n, float v0, float v1, float add0, float add1) {
      if (b2) {
        const float2 bb = __ldg(reinterpret_cast<const float2*>(b2 + n));
        v0 += bb.x;
        v1 += bb.y;
      }
      *reinterpret_cast<float2*>(yw + t * C + n) = make_float2(v0 + add0, v1 + add1);
    });
  }
}
