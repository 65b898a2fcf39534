// patch.cu -- PatchMerging / PatchSeparate of the RA-LENet U-shape, one CTA per window.
//
//   merge    (model/transformer.py:440-460): cat(x[:,0::2], x[:,1::2], -1) -> LN(2C) -> Linear(2C,2C,no bias)
//            the even/odd concat is exactly x viewed as [L/2][2C], so no gather is needed.
//   separate (model/transformer.py:418-424): 'b l (c1 c2) -> b (c1 l) c2' -> LN(C/2) -> Linear(C/2,C/2,no bias)
//            rows 0..L-1 take channels [0,C/2), rows L..2L-1 take [C/2,C); + U-skip (:650,654,658).
// Both are "rows x Cn" LayerNorm + square GEMM with rows*Cn = L*C; templated on Cn.
#define RL_NT 512        // 16 warps per window: the benchmark batch (256 windows on 148 SMs) needs the parallelism
#define RL_MINB 2
#include "common.cuh"

namespace {

// element (r, c) of the re-laid-out input inside one window
__device__ __forceinline__ int src_index(int mode, int L, int C, int Cn, int r, int c) {
  if (mode == 0) return r * Cn + c;                         // merge: contiguous view
  return (r < L) ? r * C + c : (r - L) * C + Cn + c;        // separate
}

template <int CN>
__host__ __device__ constexpr int patch_swf() {
  return cmax(WStream<CN, CN, B_NK>::FLOATS, WStream<CN, CN, B_KN>::FLOATS);
}
template <int CN>
size_t patch_smem(int rows) { return sizeof(float) * (2 * (size_t)rows * ld_mk(CN) + patch_swf<CN>() + 2 * CN + 64); }

template <int CN, int WIN>
__global__ void __launch_bounds__(RL_NT, RL_MINB) patch_fwd_kernel(const rl_patch_fwd_args a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int LDA = ld_mk(CN);
  constexpr int rows = 2048 * WIN / CN;
  const int L = a.L, C = a.C, mode = a.mode;
  float* su = smem;
  float* sw = su + 2 * rows * LDA;
  WStream<CN, CN, B_NK>::prefetch(sw, a.w, CN, nullptr, CN);   // weights do not depend on the preceding kernels
  const size_t woff = (size_t)blockIdx.x * L * C;
  if (a.skip) prefetch_l2_block(a.skip + woff, rows * CN * 4);    // nor does the U-skip tensor (written stages ago)
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  const float* xw = a.x + woff;
  {
    const float* lw = a.ln_w;
    const float* lb = a.ln_b;
    float* us = a.u ? a.u + woff : nullptr;
    // (four consecutive channels of a re-laid-out row are consecutive in the source in both modes: 16-byte accesses)
    ln_forward_rows4<CN>(
        rows, [&](int r, int c) { return ldg4(xw + src_index(mode, L, C, CN, r, c)); },
        [&](int r, int c, float4 zh) {
          const float4 u = fma4(zh, ldg4(lw + c), ldg4(lb + c));
          *reinterpret_cast<float4*>(su + r * LDA + c) = u;
          if (us) *reinterpret_cast<float4*>(us + r * CN + c) = u;
        });
  }
  __syncthreads();
  MmaTile<rows, CN> acc;
  acc.init();
  WStream<CN, CN, B_NK>::template run<true>(acc, su, LDA, sw, a.w, CN, nullptr, CN);
  const float* sk = a.skip ? a.skip + woff : nullptr;
  float* yw = a.y + woff;
  float skv[MmaTile<rows, CN>::RT][MmaTile<rows, CN>::CT][4] = {};
  if (sk) acc.gather(sk, CN, skv);                 // one batch of loads, not one round trip per element
  acc.epilogue2_pairs(skv, [&](int r, int n, float v0, float v1, float s0, float s1) {
    *reinterpret_cast<float2*>(yw + r * CN + n) = make_float2(v0 + s0, v1 + s1);
  });
}

template <int CN, int WIN, bool DET>
__global__ void __launch_bounds__(RL_NT, RL_MINB) patch_bwd_kernel(const rl_patch_bwd_args a, float* __restrict__ gsum) {
  extern __shared__ __align__(16) float smem[];
  constexpr int LDA = ld_mk(CN);
  constexpr int rows = 2048 * WIN / CN;
  const int L = a.L, C = a.C, mode = a.mode;
  float* sg = smem;
  float* su = sg + rows * LDA;
  float* sw = su + rows * LDA;
  WStream<CN, CN, B_KN>::prefetch(sw, a.w, 1 << 30, nullptr, CN);   // weights do not depend on the preceding kernels
  prefetch_l2_block(a.x + (size_t)blockIdx.x * a.L * a.C, rows * CN * 4);   // nor does the saved layer input
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  const int tid = threadIdx.x;
  const size_t woff = (size_t)blockIdx.x * L * C;
  const float* gw = a.g + woff;
  const float* g2w = a.g2 ? a.g2 + woff : nullptr;
  const float* xw = a.x + woff;
#pragma unroll
  for (int i = tid; i < rows * CN; i += RL_NT) {      // 4 (8) trips: all loads in flight together
    float v = __ldg(gw + i);
    if (g2w) {
      v += __ldg(g2w + i);
      gsum[woff + i] = v;
    }
    sg[(i / CN) * LDA + (i % CN)] = v;
  }
  __syncthreads();
  {
    MmaTile<rows, CN> acc;
    acc.init();
    WStream<CN, CN, B_KN>::template run<true>(acc, sg, LDA, sw, a.w, 1 << 30, nullptr, CN);
    acc.epilogue_pairs([&](int r, int n, float v0, float v1) {
      *reinterpret_cast<float2*>(su + r * LDA + n) = make_float2(v0, v1);
    });
  }
  __syncthreads();
  float* dxw = a.dx + woff;
  // per-warp partial rows of the LayerNorm weight / bias gradients (16 x 2CN floats): the GEMM operand tile is dead
  // (2048+ floats), at CN = 128 the weight staging area (8704 floats)
  float* s_part = (CN <= 64) ? sg : sw;
  static_assert(CN <= 64 || 32 * CN <= patch_swf<CN>(), "patch_bwd: partial rows");
  ln_backward_rows4<CN, true>(
      rows, a.ln_w, s_part, [&](int r, int c) { return ldg4(xw + src_index(mode, L, C, CN, r, c)); },
      [&](int r, int c) { return *reinterpret_cast<const float4*>(su + r * LDA + c); },
      [&](int r, int c, float4 dz, float4) { *reinterpret_cast<float4*>(dxw + src_index(mode, L, C, CN, r, c)) = dz; });
  __syncthreads();
  ln_backward_finish<CN, DET>(s_part, grad_slot<DET>(a.d_ln_w, CN, blockIdx.x), grad_slot<DET>(a.d_ln_b, CN, blockIdx.x));
}

template <int CN>
int launch_fwd(const rl_patch_fwd_args* a, cudaStream_t st) {
  const int rows = a->L * a->C / CN;
  const size_t smem = patch_smem<CN>(rows);
  if (a->L * a->C == 2048) {
    if (int rc = rl_set_smem(patch_fwd_kernel<CN, 1>, smem)) return rc;
    rl_launch_pdl(patch_fwd_kernel<CN, 1>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  } else {
    if (int rc = rl_set_smem(patch_fwd_kernel<CN, 2>, smem)) return rc;
    rl_launch_pdl(patch_fwd_kernel<CN, 2>, dim3(a->B), dim3(RL_NT), smem, st, *a);
  }
  return rl_check_launch("patch_fwd_kernel", CN);
}

template <int CN, bool DET>
int launch_bwd_det(const rl_patch_bwd_args* a, float* gsum, cudaStream_t st) {
  const int rows = a->L * a->C / CN;
  const size_t smem = patch_smem<CN>(rows);
  if (a->L * a->C == 2048) {
    if (int rc = rl_set_smem(patch_bwd_kernel<CN, 1, DET>, smem)) return rc;
    rl_launch_pdl(patch_bwd_kernel<CN, 1, DET>, dim3(a->B), dim3(RL_NT), smem, st, *a, gsum);
  } else {
    if (int rc = rl_set_smem(patch_bwd_kernel<CN, 2, DET>, smem)) return rc;
    rl_launch_pdl(patch_bwd_kernel<CN, 2, DET>, dim3(a->B), dim3(RL_NT), smem, st, *a, gsum);
  }
  return rl_check_launch("patch_bwd_kernel", CN);
}

// det: LayerNorm partials one slot per window (CTA)
template <int CN>
int launch_bwd(const rl_patch_bwd_args* a, float* gsum, cudaStream_t st, RlDet* det) {
  if (det == nullptr) return launch_bwd_det<CN, false>(a, gsum, st);
  rl_patch_bwd_args d = *a;
  d.d_ln_w = rl_det_take(det, a->d_ln_w, CN, a->B);
  d.d_ln_b = rl_det_take(det, a->d_ln_b, CN, a->B);
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "patch_bwd: deterministic-mode workspace too small");
  return launch_bwd_det<CN, true>(&d, gsum, st);
}

int check_shape(int B, int L, int C, int mode, int* cn) {
  RL_REQUIRE(B > 0 && (mode == 0 || mode == 1), RL_ERR_SHAPE, "patch: B=%d mode=%d", B, mode);
  RL_REQUIRE(L * C == 2048 || L * C == 4096, RL_ERR_SHAPE, "patch: L*C must be 2048 or 4096 (L=%d, C=%d)", L, C);
  const int CN = mode == 0 ? 2 * C : C / 2;
  RL_REQUIRE(CN == 8 || CN == 16 || CN == 32 || CN == 64 || CN == 128, RL_ERR_SHAPE, "patch: unsupported width %d", CN);
  RL_REQUIRE(mode == 1 || L % 2 == 0, RL_ERR_SHAPE, "patch: odd L=%d", L);
  *cn = CN;
  return RL_OK;
}

}  // namespace

extern "C" int ralenet_patch_fwd(const rl_patch_fwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "patch_fwd: args is NULL");
  int CN = 0;
  if (int rc = check_shape(a->B, a->L, a->C, a->mode, &CN)) return rc;
  RL_REQUIRE(a->x && a->y && a->w && a->ln_w && a->ln_b, RL_ERR_NULL, "patch_fwd: NULL tensor");
  RL_REQUIRE(rl_al16(a->x, a->y, a->w, a->ln_w, a->ln_b, a->u, a->skip), RL_ERR_SHAPE,
             "patch_fwd: tensors must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  switch (CN) {
    case 8: return launch_fwd<8>(a, st);
    case 16: return launch_fwd<16>(a, st);
    case 32: return launch_fwd<32>(a, st);
    case 64: return launch_fwd<64>(a, st);
    case 128: return launch_fwd<128>(a, st);
  }
  return RL_ERR_SHAPE;
}

// gsum: scratch [B, L*C] holding g + g2 when g2 is given (dx is used for it: see below)
// the data-gradient kernel (also leaves g + g2 in gsum for the weight gradient)
int rl_patch_bwd_main(const rl_patch_bwd_args* a, cudaStream_t st, RlDet* det) {
  RL_REQUIRE(a, RL_ERR_NULL, "patch_bwd: args is NULL");
  int CN = 0;
  if (int rc = check_shape(a->B, a->L, a->C, a->mode, &CN)) return rc;
  RL_REQUIRE(a->g && a->x && a->w && a->ln_w && a->u && a->dx, RL_ERR_NULL, "patch_bwd: NULL tensor");
  RL_REQUIRE(!a->d_ln_w == !a->d_ln_b, RL_ERR_NULL, "patch_bwd: d_ln_w/d_ln_b must be both set or both NULL");
  RL_REQUIRE(!a->g2 || a->gsum, RL_ERR_NULL, "patch_bwd: g2 needs the gsum scratch");
  RL_REQUIRE(rl_al16(a->g, a->g2, a->gsum, a->x, a->w, a->ln_w, a->u, a->dx), RL_ERR_SHAPE,
             "patch_bwd: tensors must be 16-byte aligned");
  switch (CN) {
    case 8: return launch_bwd<8>(a, a->gsum, st, det);
    case 16: return launch_bwd<16>(a, a->gsum, st, det);
    case 32: return launch_bwd<32>(a, a->gsum, st, det);
    case 64: return launch_bwd<64>(a, a->gsum, st, det);
    case 128: return launch_bwd<128>(a, a->gsum, st, det);
  }
  return RL_ERR_SHAPE;
}

bool rl_patch_bwd_has_wgrad(const rl_patch_bwd_args* a) { return a->d_w != nullptr; }

// dW = (g + g2)^T u over all tokens; may run on another stream once the main kernel is done
int rl_patch_bwd_wgrad(const rl_patch_bwd_args* a, cudaStream_t st, RlDet* det) {
  const int CN = (a->mode == 0) ? 2 * a->C : a->C / 2;
  const int M = a->B * (a->L * a->C / CN);
  const RlWgradDesc d[1] = {{a->g2 ? a->gsum : a->g, CN, a->u, CN, CN, CN, a->d_w, nullptr}};
  return rl_launch_wgrad_group(d, 1, M, st, det);
}

extern "C" int ralenet_patch_bwd(const rl_patch_bwd_args* a, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = rl_patch_bwd_main(a, st)) return rc;
  return rl_patch_bwd_wgrad(a, st);
}
