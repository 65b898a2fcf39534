// ffn.cu -- local-enhancement feed-forward half of the RA-LENet TransformerBlock, one CTA per window.
//
//   y = x + fc2( GELU( leconv( GELU( fc1( LN2(x) ) ) ) ) )  (+ extra)
//
// Reference: model/transformer.py:392-395 (forward_part2), :149-161 (Mlp.forward), :54-59
// (PartialConv_1d.forward_split_cat), :146 (depthwise variant).  As shipped the "local enhancement" is a
// 3-tap FIR along the tokens on hidden channel 0 only, followed by a second GELU on all channels
// (SURVEY.md F5); RL_LE_DEPTHWISE applies per-channel FIRs to all 4C channels; RL_LE_NONE is the plain MLP.
// The L x 4C hidden activation (8192 floats per window) stays in shared memory between the two GEMMs.
#define RL_NT 512        // 16 warps per window: the benchmark batch (256 windows on 148 SMs) needs the parallelism
#define RL_MINB 2
#include "common.cuh"

// tcgen05 kernels for the wide stages (ffn_umma.cu); return 1 when the shape/mode is not handled there
int rl_ffn_fwd_umma(const rl_ffn_fwd_args* a, cudaStream_t st);
int rl_ffn_bwd_umma(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det);

#include "ffn_body.cuh"

namespace {

template <int C, int WIN, bool TF32>
__global__ void __launch_bounds__(RL_NT, RL_MINB) ffn_fwd_kernel(const rl_ffn_fwd_args a) {
  extern __shared__ __align__(16) float smem[];
  ffn_fwd_body<C, WIN, false, TF32>(a, smem);
}

// ---------------------------------------------------------------------------------------------
// Backward.  DW = depthwise mode (needs GELU(h) of the neighbouring tokens, so it keeps the L x 4C g1 tile in
// shared memory); the shipped partial / plain modes recompute everything they need per element in the
// epilogue of the dg2 GEMM from the saved pre-activation h (one erf shared by GELU and GELU').
template <int C>
__host__ __device__ constexpr int ffn_bwd_swf() {
  // also the scratch of the in-CTA weight gradients (CtaWgrad::SCRATCH = 2304 floats) and of the per-warp LayerNorm
  // gradient partials (16 x 2C floats)
  return cmax(cmax(WStream<4 * C, C, B_KN>::FLOATS, WStream<C, 4 * C, B_KN>::FLOATS),
              cmax((C <= RL_FW_MAXC) ? 16 * 144 : 0, 32 * C));
}
// true: the fc1 / fc2 weight gradients are accumulated inside the data-gradient kernel (narrow stages, C <= 16), which
// keeps g2 in shared memory for them; false: the kernel writes g2, dh and u to the global scratch and rl_ffn_bwd_wgrad
// launches the GEMMs.  The depthwise backward of 512-sample windows (WIN = 2) already holds g1 in shared memory: with the
// g2 tile as well it would need 256 KB (C = 16) / 279 KB (C = 8), more than an SM has, so it takes the GEMM launch.
__host__ __device__ constexpr bool ffn_bwd_in_cta_wgrad(int C, int WIN, bool dw) {
  return C <= RL_FW_MAXC && !(dw && WIN == 2);
}
bool ffn_bwd_in_cta_wgrad(const rl_ffn_bwd_args* a) {
  return ffn_bwd_in_cta_wgrad(a->C, a->L * a->C / 2048, a->le_mode == RL_LE_DEPTHWISE);
}

template <int C>
size_t ffn_bwd_smem(int L, bool dw) {
  const bool fw = ffn_bwd_in_cta_wgrad(C, L * C / 2048, dw);
  return sizeof(float) * (2 * (size_t)L * ld_mk(C) + ((dw ? 2 : 1) + (fw ? 1 : 0)) * (size_t)L * ld_mk(4 * C) +
                          ffn_bwd_swf<C>() + 3 * (size_t)L + 2 * C + 64);
}

template <int C, int WIN, bool DW, bool DET>
__global__ void __launch_bounds__(RL_NT, RL_MINB) ffn_bwd_kernel(const rl_ffn_bwd_args a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int L = 2048 * WIN / C;
  constexpr int LDC = ld_mk(C);
  constexpr int HC = 4 * C, LDH = ld_mk(HC);
  float* sg = smem;                       // dL/dy, A operand
  float* su = sg + L * LDC;               // du (LN2 output gradient)
  float* sd = su + L * LDC;               // df / dh
  float* sh = sd + L * LDH;               // g1 = GELU(h), depthwise mode only
  constexpr bool FW = ffn_bwd_in_cta_wgrad(C, WIN, DW);   // weight gradients accumulated in-CTA (no wgrad launch)
  float* sg2 = sh + (DW ? L * LDH : 0);   // g2, in-CTA weight gradients only
  float* sw = sg2 + (FW ? L * LDH : 0);
  float* sg10 = sw + ffn_bwd_swf<C>();    // g1[:,0]
  float* sf0 = sg10 + L;                  // fir(g1[:,0])
  float* sdf0 = sf0 + L;                  // df[:,0]
  float* s_gb = sdf0 + L;
  float* s_red = s_gb + 2 * C;
  const int tid = threadIdx.x;
  WStream<HC, C, B_KN>::prefetch(sw, a.w2, 1 << 30, nullptr, HC);   // weights do not depend on the preceding kernels
  // neither do the tensors the forward pass saved for this window (pre-activations h, block input)
  prefetch_l2_block(a.h + (size_t)blockIdx.x * L * HC, L * HC * 4);
  prefetch_l2_block(a.x + (size_t)blockIdx.x * L * C, L * C * 4);
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  const size_t woff = (size_t)blockIdx.x * L * C;
  const size_t hoff = (size_t)blockIdx.x * L * HC;
  const float* gw = a.g + woff;
  const float* xw = a.x + woff;
  const float* hw = a.h + hoff;
  float* g2w = a.g2 + hoff;
  float* dhw = a.dh + hoff;
  const int mode = a.le_mode;

  // 1. g -> sg (asynchronously: its round trip passes behind the loads / GELUs of the cross-token pieces below);
  //    the pieces of g1 = GELU(h) that cross tokens
  for (int i = tid; i < L * (C / 4); i += RL_NT) {
    const int r = i / (C / 4), c = (i % (C / 4)) * 4;
    cp_async16(sg + r * LDC + c, gw + r * C + c);
  }
  cp_async_commit();
  float lw0 = 0.f, lw1 = 0.f, lw2 = 0.f;
  if (DW) {
    for (int i = tid; i < L * HC; i += RL_NT) sh[(i / HC) * LDH + (i % HC)] = gelu_f(__ldg(hw + i));
  } else if (mode == RL_LE_PARTIAL) {
    lw0 = __ldg(a.lew); lw1 = __ldg(a.lew + 1); lw2 = __ldg(a.lew + 2);
    for (int t = tid; t < L; t += RL_NT) sg10[t] = gelu_f(__ldg(hw + t * HC));
    __syncthreads();
    for (int t = tid; t < L; t += RL_NT) {
      const float p = (t > 0) ? sg10[t - 1] : 0.f;
      const float n = (t + 1 < L) ? sg10[t + 1] : 0.f;
      sf0[t] = lw0 * p + lw1 * sg10[t] + lw2 * n;
    }
  }
  cp_async_wait<0>();                                   // g (and the first weight chunk) have landed
  __syncthreads();
  if (DW) {   // g2 = GELU(fir(g1)) for the fc2 weight gradient
    for (int i = tid; i < L * HC; i += RL_NT) {
      const int t = i / HC, n = i % HC;
      const float p = (t > 0) ? sh[(t - 1) * LDH + n] : 0.f;
      const float nx = (t + 1 < L) ? sh[(t + 1) * LDH + n] : 0.f;
      const float g2v = gelu_f(__ldg(a.lew + 3 * n) * p + __ldg(a.lew + 3 * n + 1) * sh[t * LDH + n] +
                               __ldg(a.lew + 3 * n + 2) * nx);
      if (FW) sg2[t * LDH + n] = g2v; else g2w[i] = g2v;
    }
  }

  // 2. dg2 = g W2 (N = 4C, K = C; B(k,n) = W2[k][n] natural layout), then through GELU' / FIR^T / GELU'
  {
    MmaTile<L, HC> acc;
    acc.init();
    WStream<HC, C, B_KN>::template run<true>(acc, sg, LDC, sw, a.w2, 1 << 30, nullptr, HC);
    WStream<C, HC, B_KN>::prefetch(sw, a.w1, 1 << 30, nullptr, C);    // lands behind the GELU' / FIR-adjoint phase
    // the saved pre-activations of this thread's elements: one batch of loads (they come from HBM: a load per
    // element inside the epilogue was 16 serial round trips)
    //  (512-sample windows have 32 elements per thread: there the registers do not allow it and the loads stay inside)
    constexpr bool BATCH = MmaTile<L, HC>::TPW * 4 <= 16;
    float hv[MmaTile<L, HC>::RT][MmaTile<L, HC>::CT][4];
    if (!DW && BATCH) acc.gather(hw, HC, hv);
    if (DW) {
      acc.epilogue2(hv, [&](int t, int n, float v, float hval) {
        const float g1 = sh[t * LDH + n];
        const float p = (t > 0) ? sh[(t - 1) * LDH + n] : 0.f;
        const float nx = (t + 1 < L) ? sh[(t + 1) * LDH + n] : 0.f;
        const float f = __ldg(a.lew + 3 * n) * p + __ldg(a.lew + 3 * n + 1) * g1 + __ldg(a.lew + 3 * n + 2) * nx;
        sd[t * LDH + n] = v * gelu_grad_f(f);          // df, finished below
      });
    } else {
      // two adjacent hidden units per call: GELU / GELU' of both on the packed fp32 pipe (gelu_both2)
      acc.epilogue2_pairs(hv, [&](int t, int n, float v0, float v1, float h0, float h1) {
        if (!BATCH) { h0 = __ldg(hw + t * HC + n); h1 = __ldg(hw + t * HC + n + 1); }
        float g1[2], d1[2];
        gelu_both2(h0, h1, g1[0], g1[1], d1[0], d1[1]);
        float g2[2], dh[2];
        if (mode == RL_LE_NONE) {
          g2[0] = g1[0]; g2[1] = g1[1];
          dh[0] = v0 * d1[0]; dh[1] = v1 * d1[1];
        } else {
          // partial: the convolved channel (n == 0) takes the FIR output and is finished after the FIR adjoint,
          // the untouched channels have f == g1
          const bool conv0 = (n == 0);
          float d2[2];
          gelu_both2(conv0 ? sf0[t] : g1[0], g1[1], g2[0], g2[1], d2[0], d2[1]);
          if (conv0) sdf0[t] = v0 * d2[0];
          dh[0] = conv0 ? 0.f : v0 * d2[0] * d1[0];
          dh[1] = v1 * d2[1] * d1[1];
        }
        if (FW) *reinterpret_cast<float2*>(sg2 + t * LDH + n) = make_float2(g2[0], g2[1]);
        else *reinterpret_cast<float2*>(g2w + t * HC + n) = make_float2(g2[0], g2[1]);
        if (mode != RL_LE_NONE && n == 0) {            // (the old code left sd / dh of the convolved channel untouched)
          sd[t * LDH + 1] = dh[1];
          if (!FW) dhw[t * HC + 1] = dh[1];
        } else {
          *reinterpret_cast<float2*>(sd + t * LDH + n) = make_float2(dh[0], dh[1]);
          if (!FW) *reinterpret_cast<float2*>(dhw + t * HC + n) = make_float2(dh[0], dh[1]);
        }
      });
    }
    __syncthreads();
    if (!DW && mode == RL_LE_PARTIAL) {
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      for (int t = tid; t < L; t += RL_NT) {
        const float d = sdf0[t];
        const float dn = (t + 1 < L) ? sdf0[t + 1] : 0.f;
        const float dp = (t > 0) ? sdf0[t - 1] : 0.f;
        const float dg1 = lw0 * dn + lw1 * d + lw2 * dp;            // adjoint of the 3-tap FIR
        const float dh = dg1 * gelu_grad_f(__ldg(hw + t * HC));
        sd[t * LDH] = dh;
        if (!FW) dhw[t * HC] = dh;
        a0 += d * ((t > 0) ? sg10[t - 1] : 0.f);
        a1 += d * sg10[t];
        a2 += d * ((t + 1 < L) ? sg10[t + 1] : 0.f);
      }
      if (a.d_lew) {     // the three tap gradients: per-warp sums, ONE barrier (the one below), three threads finish
        a0 = warp_sum(a0);
        a1 = warp_sum(a1);
        a2 = warp_sum(a2);
        if ((tid & 31) == 0) { s_red[3 * (tid >> 5)] = a0; s_red[3 * (tid >> 5) + 1] = a1; s_red[3 * (tid >> 5) + 2] = a2; }
      }
      __syncthreads();
      if (a.d_lew && tid < 3) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < RL_NT / 32; ++w) s += s_red[3 * w + tid];
        grad_add<DET>(grad_slot<DET>(a.d_lew, 3, blockIdx.x) + tid, s);
      }
    } else if (DW) {
      for (int c = tid; c < HC; c += RL_NT) {
        const float w0 = __ldg(a.lew + 3 * c), w1 = __ldg(a.lew + 3 * c + 1), w2 = __ldg(a.lew + 3 * c + 2);
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
        float dprev = 0.f, dcur = sd[c];
        for (int t = 0; t < L; ++t) {
          const float dnxt = (t + 1 < L) ? sd[(t + 1) * LDH + c] : 0.f;
          const float dg1 = w0 * dnxt + w1 * dcur + w2 * dprev;
          a0 += dcur * ((t > 0) ? sh[(t - 1) * LDH + c] : 0.f);
          a1 += dcur * sh[t * LDH + c];
          a2 += dcur * ((t + 1 < L) ? sh[(t + 1) * LDH + c] : 0.f);
          const float dh = dg1 * gelu_grad_f(__ldg(hw + t * HC + c));
          sd[t * LDH + c] = dh;
          if (!FW) dhw[t * HC + c] = dh;
          dprev = dcur;
          dcur = dnxt;
        }
        if (a.d_lew) {
          float* d_lew = grad_slot<DET>(a.d_lew, 3 * HC, blockIdx.x);
          grad_add<DET>(d_lew + 3 * c, a0);
          grad_add<DET>(d_lew + 3 * c + 1, a1);
          grad_add<DET>(d_lew + 3 * c + 2, a2);
        }
      }
      __syncthreads();
    }
  }

  // 3. du = dh W1 (N = C, K = 4C; B(k,n) = W1[k][n] natural layout)
  {
    MmaTile<L, C> acc;
    acc.init();
    WStream<C, HC, B_KN>::template run<true>(acc, sd, LDH, sw, a.w1, 1 << 30, nullptr, C);
    acc.epilogue_pairs([&](int t, int n, float v0, float v1) {
      *reinterpret_cast<float2*>(su + t * LDC + n) = make_float2(v0, v1);
    });
  }
  __syncthreads();

  // 4. LN2 backward + residual
  float* dxw = a.dx + woff;
  float* uw = a.u + woff;
  const bool resid = a.flags & RL_F_RESIDUAL;
  if (a.flags & RL_F_PRENORM) {
    const float* lw = a.ln_w;
    const float* lb = a.ln_b;
    // per-warp partial rows of the LayerNorm weight / bias gradients go to the weight staging area (dead by now)
    ln_backward_rows4<C, true>(
        L, lw, sw, [&](int t, int c) { return ldg4(xw + t * C + c); },
        [&](int t, int c) { return *reinterpret_cast<const float4*>(su + t * LDC + c); },
        [&](int t, int c, float4 dz, float4 zh) {
          if (resid) {
            const float4 g4 = *reinterpret_cast<const float4*>(sg + t * LDC + c);
            dz.x += g4.x; dz.y += g4.y; dz.z += g4.z; dz.w += g4.w;
          }
          *reinterpret_cast<float4*>(dxw + t * C + c) = dz;
          // du at (t, c..c+3) was consumed by this thread
          *reinterpret_cast<float4*>(FW ? su + t * LDC + c : uw + t * C + c) = fma4(zh, ldg4(lw + c), ldg4(lb + c));
        });
    __syncthreads();
    ln_backward_finish<C, DET>(sw, grad_slot<DET>(a.d_ln_w, C, blockIdx.x), grad_slot<DET>(a.d_ln_b, C, blockIdx.x));
    if (FW) __syncthreads();                                        // sw is the weight-gradient scratch next
  } else {
    for (int i = tid; i < L * C; i += RL_NT) {
      const int t = i / C, c = i % C;
      dxw[i] = su[t * LDC + c] + (resid ? sg[t * LDC + c] : 0.f);
      if (FW) su[t * LDC + c] = __ldg(xw + i); else uw[i] = __ldg(xw + i);
    }
    __syncthreads();
  }
  if constexpr (FW) {   // dW2 = g^T g2, dW1 = dh^T u   (u now sits in su); both through the one scratch region in sw
    using W2 = CtaWgrad<C, HC, L>;
    using W1 = CtaWgrad<HC, C, L>;
    static_assert(W2::SCRATCH <= ffn_bwd_swf<C>() && W1::SCRATCH <= ffn_bwd_swf<C>(), "ffn_bwd: scratch");
    W2::partial(sg, LDC, sg2, LDH, sw);
    __syncthreads();
    W2::template reduce<DET>(sw, grad_slot<DET>(a.d_w2, C * HC, blockIdx.x), grad_slot<DET>(a.d_b2, C, blockIdx.x));
    __syncthreads();
    W1::partial(sd, LDH, su, LDC, sw);
    __syncthreads();
    W1::template reduce<DET>(sw, grad_slot<DET>(a.d_w1, HC * C, blockIdx.x), grad_slot<DET>(a.d_b1, HC, blockIdx.x));
  }
}

template <int C, bool TF32>
int launch_fwd(const rl_ffn_fwd_args* a, cudaStream_t st) {
  const size_t smem = ffn_fwd_smem<C>(a->L);
  if (a->L * C == 2048) {
    if (int rc = rl_set_smem(ffn_fwd_kernel<C, 1, TF32>, smem)) return rc;
    rl_launch_pdl(ffn_fwd_kernel<C, 1, TF32>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  } else {
    if (int rc = rl_set_smem(ffn_fwd_kernel<C, 2, TF32>, smem)) return rc;
    rl_launch_pdl(ffn_fwd_kernel<C, 2, TF32>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  }
  return rl_check_launch("ffn_fwd_kernel", C, -1, rl_tf32_tag(TF32));
}
template <int C>
int launch_fwd(const rl_ffn_fwd_args* a, cudaStream_t st) {
  return (a->flags & RL_F_TF32) ? launch_fwd<C, true>(a, st) : launch_fwd<C, false>(a, st);
}

template <int C, int WIN, bool DW, bool DET>
int launch_bwd_one(const rl_ffn_bwd_args* a, cudaStream_t st) {
  const size_t smem = ffn_bwd_smem<C>(a->L, DW);
  if (int rc = rl_set_smem(ffn_bwd_kernel<C, WIN, DW, DET>, smem)) return rc;
  rl_launch_pdl(ffn_bwd_kernel<C, WIN, DW, DET>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  return rl_check_launch("ffn_bwd_kernel", C);
}

template <int C, bool DET>
int launch_bwd_det(const rl_ffn_bwd_args* a, cudaStream_t st) {
  const bool dw = a->le_mode == RL_LE_DEPTHWISE;
  if (a->L * C == 2048) return dw ? launch_bwd_one<C, 1, true, DET>(a, st) : launch_bwd_one<C, 1, false, DET>(a, st);
  return dw ? launch_bwd_one<C, 2, true, DET>(a, st) : launch_bwd_one<C, 2, false, DET>(a, st);
}

// det: one partial slot per window (CTA) for the in-CTA gradients (LayerNorm, local enhancement; every weight where
// ffn_bwd_in_cta_wgrad)
template <int C>
int launch_bwd(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det) {
  if (det == nullptr) return launch_bwd_det<C, false>(a, st);
  rl_ffn_bwd_args d = *a;
  const int B = a->B;
  d.d_ln_w = rl_det_take(det, a->d_ln_w, C, B);
  d.d_ln_b = rl_det_take(det, a->d_ln_b, C, B);
  d.d_lew = (a->le_mode == RL_LE_NONE) ? nullptr
                                       : rl_det_take(det, a->d_lew, a->le_mode == RL_LE_DEPTHWISE ? 12 * C : 3, B);
  if (ffn_bwd_in_cta_wgrad(a)) {
    d.d_w1 = rl_det_take(det, a->d_w1, 4 * C * C, B); d.d_b1 = rl_det_take(det, a->d_b1, 4 * C, B);
    d.d_w2 = rl_det_take(det, a->d_w2, 4 * C * C, B); d.d_b2 = rl_det_take(det, a->d_b2, C, B);
  }
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "ffn_bwd: deterministic-mode workspace too small");
  return launch_bwd_det<C, true>(&d, st);
}

int check_shape(int B, int L, int C, int le) {
  RL_REQUIRE(B > 0, RL_ERR_SHAPE, "ffn: B=%d", B);
  RL_REQUIRE(C == 8 || C == 16 || C == 32 || C == 64 || C == 128, RL_ERR_SHAPE, "ffn: unsupported C=%d", C);
  RL_REQUIRE(L * C == 2048 || L * C == 4096, RL_ERR_SHAPE, "ffn: L*C must be 2048 or 4096 (L=%d, C=%d)", L, C);
  RL_REQUIRE(le >= RL_LE_NONE && le <= RL_LE_DEPTHWISE, RL_ERR_SHAPE, "ffn: bad le_mode %d", le);
  return RL_OK;
}

}  // namespace

extern "C" int ralenet_ffn_fwd(const rl_ffn_fwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "ffn_fwd: args is NULL");
  if (int rc = check_shape(a->B, a->L, a->C, a->le_mode)) return rc;
  RL_REQUIRE(a->x && a->y && a->w1 && a->w2, RL_ERR_NULL, "ffn_fwd: NULL tensor");
  RL_REQUIRE(!(a->flags & RL_F_PRENORM) || (a->ln_w && a->ln_b), RL_ERR_NULL, "ffn_fwd: prenorm needs ln");
  RL_REQUIRE(a->le_mode == RL_LE_NONE || a->lew, RL_ERR_NULL, "ffn_fwd: le_mode needs lew");
  RL_REQUIRE(!(a->flags & RL_F_TF32) || !a->h, RL_ERR_SHAPE, "ffn_fwd: RL_F_TF32 is inference only (h must be NULL)");
  RL_REQUIRE(rl_al16(a->x, a->y, a->w1, a->w2, a->ln_w, a->ln_b, a->h, a->extra), RL_ERR_SHAPE,
             "ffn_fwd: tensors must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = rl_ffn_fwd_umma(a, st);
  if (rc != 1) return rc;
  switch (a->C) {
    case 8: return launch_fwd<8>(a, st);
    case 16: return launch_fwd<16>(a, st);
    case 32: return launch_fwd<32>(a, st);
    case 64: return launch_fwd<64>(a, st);
    case 128: return launch_fwd<128>(a, st);
  }
  return RL_ERR_SHAPE;
}

int rl_ffn_bwd_main(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det) {
  RL_REQUIRE(a, RL_ERR_NULL, "ffn_bwd: args is NULL");
  RL_REQUIRE(!(a->flags & RL_F_TF32), RL_ERR_SHAPE, "ffn_bwd: RL_F_TF32 is a forward-only (inference) flag");
  if (int rc = check_shape(a->B, a->L, a->C, a->le_mode)) return rc;
  RL_REQUIRE(a->g && a->x && a->w1 && a->w2 && a->h && a->dx && a->dh && a->g2 && a->u, RL_ERR_NULL,
             "ffn_bwd: NULL tensor");
  RL_REQUIRE(!(a->flags & RL_F_PRENORM) || (a->ln_w && a->ln_b), RL_ERR_NULL, "ffn_bwd: prenorm needs ln");
  RL_REQUIRE(a->le_mode == RL_LE_NONE || a->lew, RL_ERR_NULL, "ffn_bwd: le_mode needs lew");
  RL_REQUIRE(!a->d_ln_w == !a->d_ln_b, RL_ERR_NULL, "ffn_bwd: d_ln_w/d_ln_b must be both set or both NULL");
  RL_REQUIRE(rl_al16(a->g, a->x, a->w1, a->w2, a->ln_w, a->ln_b, a->h, a->dx, a->dh, a->g2, a->u), RL_ERR_SHAPE,
             "ffn_bwd: tensors must be 16-byte aligned");
  const int rc = rl_ffn_bwd_umma(a, st, det);
  if (rc != 1) return rc;
  switch (a->C) {
    case 8: return launch_bwd<8>(a, st, det);
    case 16: return launch_bwd<16>(a, st, det);
    case 32: return launch_bwd<32>(a, st, det);
    case 64: return launch_bwd<64>(a, st, det);
    case 128: return launch_bwd<128>(a, st, det);
  }
  return RL_ERR_SHAPE;
}

bool rl_ffn_bwd_has_wgrad(const rl_ffn_bwd_args* a) { return !ffn_bwd_in_cta_wgrad(a) && (a->d_w1 || a->d_w2); }

// weight gradients from (g, g2) and (dh, u); may run on another stream once the main kernel is done
int rl_ffn_bwd_wgrad(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det) {
  const int M = a->B * a->L, C = a->C;
  if (ffn_bwd_in_cta_wgrad(a)) return RL_OK;   // accumulated inside the data-gradient kernel
  const RlWgradDesc d[2] = {{a->g, C, a->g2, 4 * C, C, 4 * C, a->d_w2, a->d_b2},
                            {a->dh, 4 * C, a->u, C, 4 * C, C, a->d_w1, a->d_b1}};
  return rl_launch_wgrad_group(d, 2, M, st, det);
}

extern "C" int ralenet_ffn_bwd(const rl_ffn_bwd_args* a, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = rl_ffn_bwd_main(a, st)) return rc;
  return rl_ffn_bwd_wgrad(a, st);
}
