// conv_mma.cu -- the lead-mixing Conv1d(k = 13, pad = 6) layers of newrale (model/ralenet_12leads.py:684-709:
// 12 -> 6 -> 2 in front of the frozen RA-LENet core, 2 -> 6 -> 12 behind it, LeakyReLU(0.01)) as IMPLICIT GEMMs on the
// tensor cores (mma.sync m16n8k8 TF32 with the 3-pass split of common.cuh, fp32-grade).  One CTA per window; the
// padded window lives in shared memory and the im2col matrix is never formed -- a fragment element A[t][(i,k)] is
// read as x[i][t + k] through a small offset table:
//
//   forward   y[t][o]   = sum_{(i,k)} x[i][t+k-6]   w[o][i][k]        M = L,    K = Cin*13 (156/78/26/78), N = Cout
//   dgrad     dx[t][i]  = sum_{(o,k)} dc[o][t-k+6]  w[o][i][k]        M = L,    K = Cout*13,               N = Cin
//   wgrad     dW[o][(i,k)] += sum_t   dc[o][t]      x[i][t+k-6]       M = Cout, K = L,                     N = Cin*13
//
// dc = dy * LeakyReLU'(pre-activation); the pre-activation is recomputed in the backward kernel by the SAME implicit
// GEMM as the forward (bit-identical sign decisions).  Channel counts are padded to the 8-wide MMA tile with zero
// weights; K to a multiple of 8.  The shapes are tiny (<= 0.5 MFLOP per window and layer), so these kernels are
// latency-bound like the rest of the 12-lead step; they exist because the north star asks for the convolutions on the
// tensor cores, and they replace the scalar FMA kernels of stem_head.cu (kept for other kernel sizes / lengths).
#define RL_NT 256
#include "common.cuh"

namespace {

constexpr int KW = 13, PAD = 6, MAXC = 12;
constexpr int KPMAX = 160;                       // padded contraction length: ceil(12 * 13 / 8) * 8
constexpr int LDB = KPMAX + 4;                   // row stride of the weight tiles (ld % 8 == 4: conflict-free B_NK)

__device__ __forceinline__ float lrelu(float v, float s) { return v > 0.f ? v : v * s; }

struct Smem {
  float* sx;      // [Ci][LP]   padded input window
  float* sdc;     // [16][LP]   gradient w.r.t. the pre-activation (rows >= Co zero), zero halo
  float* sB;      // [16][LDB]  B(kk, n) = w[n][kk], kk = i*13 + k           (forward / sign recompute)
  float* sBT;     // [16][LDB]  B(kk, i) = w[o][i][k], kk = o*13 + k          (dgrad)
  int* offA;      // [KPMAX]    (i,k) -> i*LP + k            (x gather; padding entries point at a zero row)
  int* offD;      // [KPMAX]    (o,k) -> o*LP + 12 - k       (dc gather)
};

__host__ __device__ inline size_t smem_floats(int L, int Ci, bool bwd) {
  const size_t LP = L + 2 * PAD;
  return (size_t)(Ci + 1) * LP + (bwd ? 17 * LP : 0) + (bwd ? 2 : 1) * 16 * LDB + 2 * KPMAX;
}

// acc[r][c] (+)= sum_kk src[off[kk] + t] * sB[n * LDB + kk] for the warp's two 16-row tiles and NT column tiles
template <int NT>
__device__ __forceinline__ void implicit_gemm(float (&acc)[2][NT][4], const float* __restrict__ src,
                                              const int* __restrict__ off, int KP, const float* __restrict__ sB,
                                              int row0) {
  const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  for (int k0 = 0; k0 < KP; k0 += 8) {
    const int o0 = off[k0 + t], o1 = off[k0 + t + 4];
    uint32_t ahi[2][4], alo[2][4];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int m = row0 + r * 16 + g;
      split_tf32x2(src[o0 + m], src[o0 + m + 8], ahi[r][0], ahi[r][1], alo[r][0], alo[r][1]);
      split_tf32x2(src[o1 + m], src[o1 + m + 8], ahi[r][2], ahi[r][3], alo[r][2], alo[r][3]);
    }
#pragma unroll
    for (int c = 0; c < NT; ++c) {
      const float* p = sB + (c * 8 + g) * LDB + k0 + t;
      uint32_t bhi[2], blo[2];
      split_tf32x2(p[0], p[4], bhi[0], bhi[1], blo[0], blo[1]);
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mma_tf32(acc[r][c], alo[r], bhi);
        mma_tf32(acc[r][c], ahi[r], blo);
        mma_tf32(acc[r][c], ahi[r], bhi);
      }
    }
  }
}

template <int NT>
__device__ __forceinline__ void zero_acc(float (&acc)[2][NT][4]) {
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < NT; ++c)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[r][c][e] = 0.f;
}

__device__ __forceinline__ Smem carve(float* base, int L, int Ci, bool bwd) {
  const int LP = L + 2 * PAD;
  Smem s;
  s.sx = base;
  float* p = base + (size_t)(Ci + 1) * LP;            // row Ci of sx is the all-zero row of the padding entries
  s.sdc = p;
  if (bwd) p += 17 * LP;                              // row 16 of sdc: all-zero row
  s.sB = p;
  p += 16 * LDB;
  s.sBT = p;
  if (bwd) p += 16 * LDB;
  s.offA = reinterpret_cast<int*>(p);
  s.offD = s.offA + KPMAX;
  return s;
}

// stage the padded window, the weights (zero padded to 16 x KP) and the gather table of the forward GEMM
__device__ __forceinline__ void stage_fwd(const Smem& s, const float* __restrict__ xw, const float* __restrict__ w, int L,
                                          int Ci, int Co, int KP) {
  const int LP = L + 2 * PAD, Kt = Ci * KW, tid = threadIdx.x;
  for (int i = tid; i < (Ci + 1) * LP; i += RL_NT) {
    const int ch = i / LP, p = i % LP - PAD;
    s.sx[i] = (ch < Ci && p >= 0 && p < L) ? __ldg(xw + ch * L + p) : 0.f;
  }
  for (int i = tid; i < 16 * KP; i += RL_NT) {
    const int n = i / KP, kk = i % KP;
    s.sB[n * LDB + kk] = (n < Co && kk < Kt) ? __ldg(w + n * Kt + kk) : 0.f;
  }
  for (int kk = tid; kk < KP; kk += RL_NT) s.offA[kk] = kk < Kt ? (kk / KW) * LP + kk % KW : Ci * LP;
}

// pre-activation tile of this warp: s[t][o] = b[o] + sum x w
template <int NT>
__device__ __forceinline__ void preact(float (&acc)[2][NT][4], const Smem& s, int KP, int row0) {
  zero_acc<NT>(acc);
  implicit_gemm<NT>(acc, s.sx, s.offA, KP, s.sB, row0);
}

template <int NT>
__global__ void __launch_bounds__(RL_NT) conv13_fwd_mma_kernel(const rl_conv_fwd_args a) {
  extern __shared__ __align__(16) float smem[];
  const int L = a.L, Ci = a.Cin, Co = a.Cout, KP = (Ci * KW + 7) & ~7;
  const Smem s = carve(smem, L, Ci, false);
  stage_fwd(s, a.x + (size_t)blockIdx.x * Ci * L, a.w, L, Ci, Co, KP);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  float* yw = a.y + (size_t)blockIdx.x * Co * L;
  for (int row0 = warp * 32; row0 < L; row0 += (RL_NT / 32) * 32) {
    float acc[2][NT][4];
    preact<NT>(acc, s, KP, row0);
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int c = 0; c < NT; ++c)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int m = row0 + r * 16 + g + (e >> 1) * 8, o = c * 8 + 2 * t + (e & 1);
          if (o < Co) {
            const float v = acc[r][c][e] + (a.b ? __ldg(a.b + o) : 0.f);
            yw[o * L + m] = a.act ? lrelu(v, a.slope) : v;
          }
        }
  }
}

// DET: d_w / d_b are partial slabs [B][Cout*Cin*13] / [B][Cout] (grad_add): every element of a window's dW is one
// element of one warp tile, every element of its db the sum of one warp, so the slot of a CTA is its window
template <int NTO, int NTI, bool DET>     // column tiles of the forward GEMM (Cout) and of the dgrad GEMM (Cin)
__global__ void __launch_bounds__(RL_NT) conv13_bwd_mma_kernel(const rl_conv_bwd_args a) {
  extern __shared__ __align__(16) float smem[];
  const int L = a.L, Ci = a.Cin, Co = a.Cout, LP = L + 2 * PAD;
  const int KP = (Ci * KW + 7) & ~7, KPD = (Co * KW + 7) & ~7, Kt = Ci * KW;
  const Smem s = carve(smem, L, Ci, true);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  stage_fwd(s, a.x + (size_t)blockIdx.x * Ci * L, a.w, L, Ci, Co, KP);
  for (int i = tid; i < 17 * LP; i += RL_NT) s.sdc[i] = 0.f;
  for (int i = tid; i < 16 * KPD; i += RL_NT) {      // B(kk = (o,k), n = i) = w[o][i][k]
    const int n = i / KPD, kk = i % KPD, o = kk / KW, k = kk % KW;
    s.sBT[n * LDB + kk] = (n < Ci && kk < Co * KW) ? __ldg(a.w + (o * Ci + n) * KW + k) : 0.f;
  }
  for (int kk = tid; kk < KPD; kk += RL_NT) s.offD[kk] = kk < Co * KW ? (kk / KW) * LP + 2 * PAD - kk % KW : 16 * LP;
  __syncthreads();

  // 1. dc[o][t] = dy[o][t] * LeakyReLU'(pre-activation), pre-activation recomputed exactly as the forward does
  const float* dyw = a.dy + (size_t)blockIdx.x * Co * L;
  for (int row0 = warp * 32; row0 < L; row0 += (RL_NT / 32) * 32) {
    float acc[2][NTO][4];
    if (a.act) preact<NTO>(acc, s, KP, row0);
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
      for (int c = 0; c < NTO; ++c)
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int m = row0 + r * 16 + g + (e >> 1) * 8, o = c * 8 + 2 * t + (e & 1);
          if (o < Co) {
            float d = __ldg(dyw + o * L + m);
            if (a.act) {
              const float v = acc[r][c][e] + (a.b ? __ldg(a.b + o) : 0.f);
              if (!(v > 0.f)) d *= a.slope;
            }
            s.sdc[o * LP + PAD + m] = d;
          }
        }
  }
  __syncthreads();

  // 2. dgrad: dx[i][t] = sum_{(o,k)} dc[o][t + 12 - k - 6] w[o][i][k]   (sdc row offset PAD is folded into offD)
  if (a.dx) {
    float* dxw = a.dx + (size_t)blockIdx.x * Ci * L;
    for (int row0 = warp * 32; row0 < L; row0 += (RL_NT / 32) * 32) {
      float acc[2][NTI][4];
      zero_acc<NTI>(acc);
      implicit_gemm<NTI>(acc, s.sdc, s.offD, KPD, s.sBT, row0);
#pragma unroll
      for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < NTI; ++c)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const int m = row0 + r * 16 + g + (e >> 1) * 8, i = c * 8 + 2 * t + (e & 1);
            if (i < Ci) dxw[i * L + m] = acc[r][c][e];
          }
    }
  }

  // 3. wgrad: dW[o][(i,k)] += sum_t dc[o][t] x[i][t+k-6]: one 16 x 8 tile of dW per warp step, K = L
  if (a.d_w) {
    float* const d_w = grad_slot<DET>(a.d_w, (size_t)Co * Kt, blockIdx.x);
    for (int nt = warp; nt < KP / 8; nt += RL_NT / 32) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      const int ob = s.offA[nt * 8 + g];                    // B(k = t', n = (i,k)) = x[i][t' + k]
      for (int k0 = 0; k0 < L; k0 += 8) {
        uint32_t ahi[4], alo[4], bhi[2], blo[2];
        split_tf32x2(s.sdc[g * LP + PAD + k0 + t], s.sdc[(g + 8) * LP + PAD + k0 + t], ahi[0], ahi[1], alo[0], alo[1]);
        split_tf32x2(s.sdc[g * LP + PAD + k0 + t + 4], s.sdc[(g + 8) * LP + PAD + k0 + t + 4], ahi[2], ahi[3], alo[2], alo[3]);
        split_tf32x2(s.sx[ob + k0 + t], s.sx[ob + k0 + t + 4], bhi[0], bhi[1], blo[0], blo[1]);
        mma_tf32(acc, alo, bhi);
        mma_tf32(acc, ahi, blo);
        mma_tf32(acc, ahi, bhi);
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int o = g + (e >> 1) * 8, n = nt * 8 + 2 * t + (e & 1);
        if (o < Co && n < Kt) grad_add<DET>(d_w + o * Kt + n, acc[e]);
      }
    }
    if (a.d_b) {
      float* const d_b = grad_slot<DET>(a.d_b, Co, blockIdx.x);
      for (int o = warp; o < Co; o += RL_NT / 32) {
        float sum = 0.f;
        for (int m = lane; m < L; m += 32) sum += s.sdc[o * LP + PAD + m];
#pragma unroll
        for (int sft = 16; sft > 0; sft >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, sft);
        if (lane == 0) grad_add<DET>(d_b + o, sum);
      }
    }
  }
}

int g_conv_mma = -1;
int conv_mma_on() {
  if (g_conv_mma < 0) {
    const char* e = getenv("RALENET_CONV_MMA");
    g_conv_mma = (e && e[0] == '0') ? 0 : 1;
  }
  return g_conv_mma;
}

}  // namespace

extern "C" int ralenet_set_conv_mma(int on) {
  const int prev = conv_mma_on();
  g_conv_mma = on ? 1 : 0;
  return prev;
}

bool rl_conv13_eligible(int L, int Ci, int Co, int K) {
  return conv_mma_on() && K == KW && L % 32 == 0 && L <= 1024 && Ci <= MAXC && Co <= MAXC && Ci > 0 && Co > 0;
}

int rl_conv13_fwd_mma(const rl_conv_fwd_args* a, cudaStream_t st) {
  const size_t smem = sizeof(float) * smem_floats(a->L, a->Cin, false);
  rl_prof_pre(st);
  if (a->Cout <= 8) {
    if (int rc = rl_set_smem(conv13_fwd_mma_kernel<1>, smem)) return rc;
    conv13_fwd_mma_kernel<1><<<a->B, RL_NT, smem, st>>>(*a);
  } else {
    if (int rc = rl_set_smem(conv13_fwd_mma_kernel<2>, smem)) return rc;
    conv13_fwd_mma_kernel<2><<<a->B, RL_NT, smem, st>>>(*a);
  }
  return rl_check_launch("conv13_fwd_mma_kernel", a->Cin, a->Cout);
}

template <int NTO, int NTI, bool DET>
static int launch_bwd(const rl_conv_bwd_args* a, size_t smem, cudaStream_t st) {
  if (int rc = rl_set_smem(conv13_bwd_mma_kernel<NTO, NTI, DET>, smem)) return rc;
  conv13_bwd_mma_kernel<NTO, NTI, DET><<<a->B, RL_NT, smem, st>>>(*a);
  return RL_OK;
}

template <bool DET>
static int launch_bwd(const rl_conv_bwd_args* a, size_t smem, cudaStream_t st) {
  if (a->Cout <= 8) return a->Cin <= 8 ? launch_bwd<1, 1, DET>(a, smem, st) : launch_bwd<1, 2, DET>(a, smem, st);
  return a->Cin <= 8 ? launch_bwd<2, 1, DET>(a, smem, st) : launch_bwd<2, 2, DET>(a, smem, st);
}

int rl_conv13_bwd_mma(const rl_conv_bwd_args* a, cudaStream_t st, bool det) {
  const size_t smem = sizeof(float) * smem_floats(a->L, a->Cin, true);
  rl_prof_pre(st);
  if (int rc = det ? launch_bwd<true>(a, smem, st) : launch_bwd<false>(a, smem, st)) return rc;
  return rl_check_launch("conv13_bwd_mma_kernel", a->Cin, a->Cout);
}
