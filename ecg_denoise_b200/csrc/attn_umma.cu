// attn_umma.cu -- attention half for the WIDE stages (C = 64, 128) with both projections on the 5th-generation
// tensor cores (tcgen05.mma kind::tf32, accumulators in tensor memory); forward only.
//
//   y = x + proj( softmax(0.5 q k^T + rw_bias) v ),   [q | k | v] = LN1(x*sqrt(C) + P) [Wq ; Wkv]^T + b
//
// Same arithmetic as attn.cu (reference model/transformer.py:383-390, 289-323, 226-247, 179-181, 534-558).
//
// At the wide stages a window has only L = 32 / 16 tokens while attn_fwd_kernel streams 64 / 256 KB of weights
// through every one-window CTA (profiles/r1_v7_trace_attn.txt: the kernel is L2 -> SM weight traffic).  Here a tile
// of TM = 128 tokens = 4 / 8 whole windows forms the M dimension of the UMMAs and a cluster of NSL = C / 32 CTAs
// SPLITS THE HEADS: CTA r owns the 8 heads [8 r, 8 r + 8) = channels [32 r, 32 r + 32) of q, k and v:
//   1. PE + LN1 of the 128 tokens -> A tile (K-major) with tf32 remainders          (every CTA of the cluster)
//   2. [q | k | v] slice = u [Wq_r ; Wk_r ; Wv_r]^T     UMMA M = 128, N = 96, K = C  -> TMEM columns [0, 96)
//   3. TMEM -> shared memory (+ bias, saved for the backward), attention core of the 8 heads of the 4 / 8 windows
//      on mma.sync (attn_core.cuh: head_dim 4 has no UMMA shape), one (window, head, 16-query tile) per warp
//   4. partial projection  yp = o_r Wp[:, 32 r : 32 r + 32]^T    UMMA M = 128, N = C, K = 32 -> TMEM columns [96, 96 + C)
//   5. the NSL partial tiles are reduced through distributed shared memory; + bias + residual -> y
// so a CTA reads 96 C + 32 C weights for 128 tokens instead of 4 C^2 per window (32x less L2 -> SM traffic at C = 128).
// Operand staging, the 3-pass tf32 split and completion tracking are those of ffn_umma.cu (umma.cuh).
#define RL_NT 512
#define RL_MINB 1
#include "common.cuh"
#include "attn_core.cuh"
#include "umma.cuh"
#include "tma.cuh"
#include <cooperative_groups.h>
#include <stdlib.h>

namespace cg = cooperative_groups;

#ifndef RL_ATTN_UMMA_DEFAULT
#define RL_ATTN_UMMA_DEFAULT 1   // see ralenet_set_attn_umma() below
#endif

RL_TRACE_DEFINE(attn_umma)

namespace {

constexpr int TM = 128;          // tokens per tile (UMMA M)
constexpr int CS = 32;           // channels (8 heads) per CTA
constexpr int NQ = 3 * CS;       // UMMA N of the [q | k | v] slice
constexpr int KC = 32;           // contraction chunk staged per pipeline step
constexpr int LDS = CS + 4;      // row stride of the q / k / v slices in shared memory (ld_mk(32): conflict-free)
constexpr int TMEM_COLS = 256;
using umma::Ring;

template <int C>
struct ASmem {
  // region 0: u tile (hi | lo) -> q, k, v slices [TM][LDS] -> partial projection tile [TM][C + 4]
  static constexpr int R0 = cmax(cmax(2 * TM * C, 3 * TM * LDS), TM * (C + 4));
  // region 1: weight ring of the q|k|v GEMM (2 stages x (hi | lo)) -> o tile (hi | lo) + Wp slice (hi | lo)
  static constexpr int R1 = cmax(4 * NQ * KC, 2 * TM * CS + 2 * C * CS);
  // constants staged before the dependency wait: positional tile [L][C + 4] (L * C = 2048), norm1 weight | bias
  static constexpr int LDPE = C + 4;
  static constexpr int CONSTS = (2048 / C) * LDPE + 2 * C;
  static constexpr size_t BYTES = sizeof(float) * (R0 + R1 + 128 + CONSTS) + 64;
};

// The weight operands arrive through cp.async.bulk.tensor (tma.cuh): per 32-wide K chunk three 32-row boxes (the q, k
// and v rows of this CTA's head slice, from to_q and the two halves of to_kv) into one 96-row SWIZZLE_128B tile, and one
// C-row box for the K-slice of the output projection.  TF32 (RL_F_TF32): single-pass projection MMAs on operand tiles
// rounded to tf32 (no remainder tiles); the attention core is the same in both forms.
template <int C, bool TF32>
__global__ void __launch_bounds__(RL_NT, RL_MINB) attn_fwd_umma_kernel(const rl_attn_fwd_args a,
                                                                       const __grid_constant__ CUtensorMap tmq,
                                                                       const __grid_constant__ CUtensorMap tmkv,
                                                                       const __grid_constant__ CUtensorMap tmp) {
  constexpr int L = 2048 / C, H = C / RL_HD, NSL = C / CS, NWT = TM / L, HS = CS / RL_HD, QT = L / 16;
  constexpr int NCHK = C / KC;
  extern __shared__ __align__(1024) float smem[];
  float* r0 = smem;
  float* r1 = smem + ASmem<C>::R0;
  float* stab = r1 + ASmem<C>::R1;                           // R-wave table * log2(e), (2W-1) x H <= 128 floats
  float* s_pe = stab + 128;                                  // positional tile [L][LDPE]
  float* s_ln = s_pe + L * ASmem<C>::LDPE;                   // norm1 weight [C] | bias [C]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_ln + 2 * C);   // [0,1] MMAs of a ring buffer done, [2,3] q|k|v chunk
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);  // landed, [4] Wp slice landed
  const int r_early = (int)(blockIdx.x % NSL);
  auto tma_issue_qkv = [&](int j) {      // tid 0: chunk j of [Wq_r ; Wk_r ; Wv_r] -> ring buffer j & 1 (hi tile)
    float* dst = r1 + (j & 1) * 2 * NQ * KC;
    uint64_t* bar = bars + 2 + (j & 1);
    tma::expect_tx(bar, NQ * KC * 4);
    tma::load_2d(dst, &tmq, j * KC, CS * r_early, bar);
    tma::load_2d(dst + CS * KC, &tmkv, j * KC, CS * r_early, bar);
    tma::load_2d(dst + 2 * CS * KC, &tmkv, j * KC, C + CS * r_early, bar);
  };
  if (threadIdx.x == 0) {
    umma::mbar_init(bars, 1);
    umma::mbar_init(bars + 1, 1);
    umma::mbar_init(bars + 2, 1);
    umma::mbar_init(bars + 3, 1);
    umma::mbar_init(bars + 4, 1);
    umma::fence_mbar_init();
    umma::fence_async_smem();
    tma::prefetch_desc(&tmq);
    tma::prefetch_desc(&tmkv);
    tma::prefetch_desc(&tmp);
    tma_issue_qkv(0);                    // weights are immutable inside the step: the ring fills while the previous
    tma_issue_qkv(1);                    // kernel drains (NCHK >= 2)
  }
  // ... and so do the constants of phase 1 (positional tile, LayerNorm affine) and the R-wave table: staged in
  // shared memory here, phase 1 then waits for ONE round of global loads (x) instead of three
  {
    constexpr int LDPE = ASmem<C>::LDPE;
    const int t = threadIdx.x;
    if (a.flags & RL_F_PRENORM) {
      static_assert(L * C / 4 == RL_NT, "one float4 of the positional tile per thread");
      const float4 p4 = __ldg(reinterpret_cast<const float4*>(a.pe) + t);
      float4 l4 = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < C / 2) l4 = __ldg(reinterpret_cast<const float4*>(t < C / 4 ? a.ln_w : a.ln_b) + (t % (C / 4)));
      *reinterpret_cast<float4*>(s_pe + (t / (C / 4)) * LDPE + 4 * (t % (C / 4))) = p4;
      if (t < C / 2) *reinterpret_cast<float4*>(s_ln + 4 * t) = l4;
    }
    if (a.W > 0 && t < (2 * a.W - 1) * H) stab[t] = __ldg(a.table + t) * RL_LOG2E;   // (2W-1) x H <= 128 entries
  }
  RL_TS(attn_umma, 0);
  pdl_wait();
  pdl_trigger();
  RL_TS(attn_umma, 1);
  float* sA_hi = r0;                                         // u tile, K-major, KT = C
  float* sA_lo = r0 + TM * C;
  float* sq = r0;                                            // q, k, v slices [TM][LDS] (over the dead u tile)
  float* sk = sq + TM * LDS;
  float* sv = sk + TM * LDS;
  float* sB = r1;                                            // [2 stages][hi | lo][NQ * KC]
  float* sO_hi = r1;                                         // o tile, K-major, KT = CS (over the dead ring)
  float* sO_lo = sO_hi + TM * CS;
  float* sW_hi = sO_lo + TM * CS;                            // Wp[:, 32 r : 32 r + 32], K-major, KT = CS
  float* sW_lo = sW_hi + C * CS;

  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int tile = blockIdx.x / NSL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t tok0 = (size_t)tile * TM;
  const int nvalid = min(TM, a.B * L - (int)tok0);            // valid token rows of this tile (whole windows)
  const float* xw = a.x + tok0 * C;
  const int W = a.W, c0 = a.c0;

  if (warp == 0) umma::tmem_alloc<TMEM_COLS>(tmem_slot);
  __syncthreads();                                           // staged constants visible to every warp
  RL_TS(attn_umma, 2);

  // 1. x*sqrt(C) + P -> LayerNorm -> A tile (K-major, KT = C) with its tf32 remainder     (transformer.py:386-387)
  //    A warp owns 8 rows; lane = (row % 8, 16-byte chunk % 4): full sectors from global, contiguous tile stores.
  {
    constexpr int NI = C / 16;                                // chunks per lane
    const int rsub = lane & 7, qsub = lane >> 3;
    const int row = warp * 8 + rsub;
    const bool ok = row < nvalid;
    const bool pre = a.flags & RL_F_PRENORM;
    const float sc = sqrtf((float)C);
    float4 v[NI];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int qc = qsub + 4 * i;
      v[i] = ok ? __ldg(reinterpret_cast<const float4*>(xw + (size_t)row * C) + qc) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (pre) {
        const float4 p4 = *reinterpret_cast<const float4*>(s_pe + (row % L) * ASmem<C>::LDPE + 4 * qc);
        v[i].x = fmaf(v[i].x, sc, p4.x); v[i].y = fmaf(v[i].y, sc, p4.y);
        v[i].z = fmaf(v[i].z, sc, p4.z); v[i].w = fmaf(v[i].w, sc, p4.w);
      }
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    RL_TS(attn_umma, 13);                                     // (trace) the x loads have landed
    float mu = 0.f, rstd = 1.f;
    if (pre) {
      s += __shfl_xor_sync(0xffffffffu, s, 8);
      s += __shfl_xor_sync(0xffffffffu, s, 16);
      mu = s * (1.0f / C);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < NI; ++i) {
        const float d0 = v[i].x - mu, d1 = v[i].y - mu, d2 = v[i].z - mu, d3 = v[i].w - mu;
        q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
      }
      q += __shfl_xor_sync(0xffffffffu, q, 8);
      q += __shfl_xor_sync(0xffffffffu, q, 16);
      rstd = rsqrtf(q * (1.0f / C) + RL_LN_EPS);
    }
    RL_TS(attn_umma, 14);                                     // (trace) statistics done
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int qc = qsub + 4 * i;
      float4 u = v[i];
      if (pre) {
        const float4 w4 = *reinterpret_cast<const float4*>(s_ln + 4 * qc);
        const float4 b4 = *reinterpret_cast<const float4*>(s_ln + C + 4 * qc);
        u.x = fmaf((v[i].x - mu) * rstd, w4.x, b4.x);
        u.y = fmaf((v[i].y - mu) * rstd, w4.y, b4.y);
        u.z = fmaf((v[i].z - mu) * rstd, w4.z, b4.z);
        u.w = fmaf((v[i].w - mu) * rstd, w4.w, b4.w);
      }
      if (!ok) u = make_float4(0.f, 0.f, 0.f, 0.f);
      const int o = rsub * 4 + qc * 32 + warp * (C / 4) * 32;
      if constexpr (TF32) {
        *reinterpret_cast<float4*>(sA_hi + o) = umma::rna4(u);
      } else {
        *reinterpret_cast<float4*>(sA_hi + o) = u;
        *reinterpret_cast<float4*>(sA_lo + o) = umma::lo4(u);
      }
    }
  }
  umma::tc_fence_before();
  __syncthreads();
  umma::tc_fence_after();
  const uint32_t tb = *tmem_slot;
  Ring ring{bars, 0};
  RL_TS(attn_umma, 3);

  // 2. [q | k | v] slice = u [Wq_r ; Wk_r ; Wv_r]^T   (M = TM, N = NQ, K = C) -> TMEM columns [0, NQ)
  {
    constexpr uint32_t idesc = umma::idesc_tf32(TM, NQ);
#pragma unroll
    for (int j = 0; j < NCHK; ++j) {
      float* bh = sB + ring.buf() * 2 * NQ * KC;
      float* bl = bh + NQ * KC;
      umma::mbar_wait(bars + 2 + (j & 1), (uint32_t)((j >> 1) & 1));
      tma::derive_lo<RL_NT, TF32>(bh, bl, NQ * KC);
      umma::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        umma::tc_fence_after();
        tma::mma_chunk_3x<KC, TF32>(tb, sA_hi, sA_lo, C, j * KC, bh, bl, idesc, j > 0 ? 1u : 0u);
        umma::commit(bars + ring.buf());
        if (j + 2 < NCHK) {              // refill this buffer once its MMAs have drained
          ++ring.chunk;
          ring.wait_last();
          --ring.chunk;
          tma_issue_qkv(j + 2);
        }
      }
      ++ring.chunk;
    }
  }
  // the bias values of epilogue 1 go to registers now; their latency hides behind the MMAs (warp group w / 4 = 0, 1, 2
  // takes q, k, v)
  float4 bias4[CS / 4];
  {
    const int seg = warp >> 2;
    const float* bias = (seg == 0) ? a.bq : a.bkv;
#pragma unroll
    for (int i = 0; i < CS / 4; ++i) bias4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (seg < 3 && bias) {
      bias += ((seg == 2) ? C : 0) + CS * r;
#pragma unroll
      for (int i = 0; i < CS / 4; ++i) bias4[i] = __ldg(reinterpret_cast<const float4*>(bias) + i);
    }
  }
  RL_TS(attn_umma, 4);
  ring.wait_last();
  umma::tc_fence_after();
  RL_TS(attn_umma, 5);
  // the ring is dead (its last MMAs have completed): the K-slice Wp[:, 32 r : 32 r + 32] lands over it while
  // epilogue 1 and the attention core run
  if (tid == 0) {
    tma::expect_tx(bars + 4, C * CS * 4);
    tma::load_2d(sW_hi, &tmp, CS * r, 0, bars + 4);
  }

  // 3a. epilogue 1: + bias, q / k / v slices -> shared memory [TM][LDS] (over the dead u tile) and, for the
  //     backward, global memory.  Warp w reads TMEM lane quadrant w % 4; warp group w / 4 = 0, 1, 2 takes q, k, v.
  {
    const int quad = warp & 3, seg = warp >> 2;
    const int row = quad * 32 + lane;
    if (seg < 3) {
      float hv[32];
      {
        float t0[16], t1[16];
        umma::tmem_ld16(umma::tmem_addr(tb, seg * CS), t0);
        umma::tmem_ld16(umma::tmem_addr(tb, seg * CS + 16), t1);
#pragma unroll
        for (int i = 0; i < 16; ++i) { hv[i] = t0[i]; hv[16 + i] = t1[i]; }
      }
#pragma unroll
      for (int i = 0; i < CS / 4; ++i) {
        hv[4 * i] += bias4[i].x; hv[4 * i + 1] += bias4[i].y; hv[4 * i + 2] += bias4[i].z; hv[4 * i + 3] += bias4[i].w;
      }
      float4* dst = reinterpret_cast<float4*>(r0 + seg * TM * LDS + row * LDS);
#pragma unroll
      for (int i = 0; i < 8; ++i) dst[i] = make_float4(hv[4 * i], hv[4 * i + 1], hv[4 * i + 2], hv[4 * i + 3]);
    }
  }
  umma::tc_fence_before();     // the tcgen05.ld reads of the q|k|v accumulator precede the barrier below
  __syncthreads();
  // q, k, v slices -> global memory for the backward: 8 lanes cover the 128 contiguous bytes of one token, so a warp
  // writes four full lines per store (one thread per row, as the accumulator is read, would touch 32 lines)
  if (a.q) {
#pragma unroll
    for (int it = 0; it < 3 * TM * (CS / 4) / RL_NT; ++it) {
      const int idx = tid + it * RL_NT;
      const int seg = idx / (TM * (CS / 4)), row = (idx / (CS / 4)) % TM, c4 = idx % (CS / 4);
      if (row < nvalid) {
        float* gsave = (seg == 0) ? a.q : (seg == 1) ? a.k : a.v;
        *reinterpret_cast<float4*>(gsave + (tok0 + row) * C + CS * r + 4 * c4) =
            *reinterpret_cast<const float4*>(r0 + seg * TM * LDS + row * LDS + 4 * c4);
      }
    }
    __syncthreads();           // q is overwritten by o below
  }
  RL_TS(attn_umma, 6);

  // 3b. attention core of the HS heads of the NWT windows: one (window, head, 16-query tile) item per warp
  //     (attn_core.cuh); o overwrites q in place.  Windows attend only within themselves.
  {
    const int nwin = nvalid / L;
    constexpr int NITEM = NWT * HS * QT;
#pragma unroll 1
    for (int item = warp; item < NITEM; item += RL_NT / 32) {
      const int w = item / (HS * QT), h = (item / QT) % HS, i0 = (item % QT) * 16;
      if (w >= nwin) continue;
      const int hg = HS * r + h;                              // head index within the layer
      attn_core_fwd_item<L, LDS>(sq + w * L * LDS, sk + w * L * LDS, sv + w * L * LDS, 4 * h, i0, stab + hg, H, W, c0,
                                 a.lse ? a.lse + ((size_t)(tile * NWT + w) * H + hg) * L : nullptr);
    }
  }
  __syncthreads();
  RL_TS(attn_umma, 7);

  // 4. o slice -> A tile (K-major, KT = CS) with remainder (+ global copy for the backward), Wp slice -> B tile;
  //    partial projection yp = o_r Wp[:, 32 r : 32 r + 32]^T  (M = TM, N = C, K = CS) -> TMEM columns [NQ, NQ + C)
  {
    const int rsub = lane & 7, qsub = lane >> 3;
    const int row = warp * 8 + rsub;
#pragma unroll
    for (int i = 0; i < CS / 16; ++i) {
      const int qc = qsub + 4 * i;
      const float4 o4 = *reinterpret_cast<const float4*>(sq + row * LDS + 4 * qc);
      if (a.o && row < nvalid) *reinterpret_cast<float4*>(a.o + (tok0 + row) * C + CS * r + 4 * qc) = o4;
      const int o = rsub * 4 + qc * 32 + warp * (CS / 4) * 32;
      if constexpr (TF32) {
        *reinterpret_cast<float4*>(sO_hi + o) = umma::rna4(o4);
      } else {
        *reinterpret_cast<float4*>(sO_hi + o) = o4;
        *reinterpret_cast<float4*>(sO_lo + o) = umma::lo4(o4);
      }
    }
    umma::mbar_wait(bars + 4, 0u);
    tma::derive_lo<RL_NT, TF32>(sW_hi, sW_lo, C * CS);
    umma::fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      constexpr uint32_t idesc = umma::idesc_tf32(TM, C);
      umma::tc_fence_after();
      tma::mma_chunk_3x<CS, TF32>(tb + NQ, sO_hi, sO_lo, CS, 0, sW_hi, sW_lo, idesc, 0u);
      umma::commit(bars + ring.buf());
    }
    ++ring.chunk;
  }
  ring.wait_last();
  umma::tc_fence_after();
  RL_TS(attn_umma, 8);

  // 5. epilogue 2: partial tile -> shared memory [TM][C + 4] (over the dead q / k / v slices), DSMEM reduction:
  //    CTA r finishes rows [r * TM / NSL, (r + 1) * TM / NSL)        y = x + o Wp^T + bp  (transformer.py:320, :405)
  constexpr int LDP = C + 4;
  float* sp = r0;
  {
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    constexpr int CW = C / 4;                                 // columns per warp group (16 or 32)
#pragma unroll
    for (int c16 = 0; c16 < CW; c16 += 16) {
      float t0[16];
      umma::tmem_ld16(umma::tmem_addr(tb, NQ + cgp * CW + c16), t0);
#pragma unroll
      for (int i = 0; i < 16; i += 4)
        *reinterpret_cast<float4*>(sp + row * LDP + cgp * CW + c16 + i) = make_float4(t0[i], t0[i + 1], t0[i + 2], t0[i + 3]);
    }
  }
  umma::tc_fence_before();
  // rows [r RPC, (r + 1) RPC) are finished here: their bias + residual terms are fetched before the cluster barrier
  constexpr int RPC = TM / NSL, RIT = RPC * (C / 4) / RL_NT;  // rows finished by this CTA, float4 items per thread
  static_assert(RPC * (C / 4) % RL_NT == 0, "reduce: items must tile the CTA");
  float4 add4[RIT];
#pragma unroll
  for (int it = 0; it < RIT; ++it) {
    const int i = tid + it * RL_NT;
    const int rr = r * RPC + i / (C / 4), c = (i % (C / 4)) * 4;
    add4[it] = a.bp ? __ldg(reinterpret_cast<const float4*>(a.bp + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if ((a.flags & RL_F_RESIDUAL) && rr < nvalid) {
      const float4 x4 = __ldg(reinterpret_cast<const float4*>(a.x + (tok0 + rr) * C + c));
      add4[it].x += x4.x; add4[it].y += x4.y; add4[it].z += x4.z; add4[it].w += x4.w;
    }
  }
  RL_TS(attn_umma, 9);
  cluster.sync();
  RL_TS(attn_umma, 10);
  {
    const float* part[NSL];
#pragma unroll
    for (int q = 0; q < NSL; ++q) part[q] = cluster.map_shared_rank(sp, q);
#pragma unroll
    for (int it = 0; it < RIT; ++it) {
      const int i = tid + it * RL_NT;
      const int rr = r * RPC + i / (C / 4), c = (i % (C / 4)) * 4;
      if (rr >= nvalid) continue;
      const int off = rr * LDP + c;
      float4 s = *reinterpret_cast<const float4*>(part[0] + off);
#pragma unroll
      for (int q = 1; q < NSL; ++q) {
        const float4 p = *reinterpret_cast<const float4*>(part[q] + off);
        s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
      }
      s.x += add4[it].x; s.y += add4[it].y; s.z += add4[it].z; s.w += add4[it].w;
      *reinterpret_cast<float4*>(a.y + (tok0 + rr) * C + c) = s;
    }
  }
  RL_TS(attn_umma, 11);
  cluster.sync();     // nobody may exit while its partial tile is still being read
  if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tb);
  RL_TS(attn_umma, 12);
}

template <int C, bool TF32>
int launch(const rl_attn_fwd_args& a, cudaStream_t st) {
  constexpr int NSL = C / CS;
  const int tiles = (a.B * a.L + TM - 1) / TM;
  CUtensorMap tmq = {}, tmkv = {}, tmp = {};
  if (int rc = rl_tmap_weight(a.wq, C, C, C, CS, &tmq)) return rc;            // to_q  [C][C]:  32-row boxes
  if (int rc = rl_tmap_weight(a.wkv, 2 * C, C, C, CS, &tmkv)) return rc;      // to_kv [2C][C]: 32-row boxes
  if (int rc = rl_tmap_weight(a.wp, C, C, C, C, &tmp)) return rc;             // proj  [C][C]:  all C rows, 32 columns
  auto kernel = attn_fwd_umma_kernel<C, TF32>;
  if (int rc = rl_set_smem(kernel, ASmem<C>::BYTES)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(tiles * NSL);
  cfg.blockDim = dim3(RL_NT);
  cfg.dynamicSmemBytes = ASmem<C>::BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = NSL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  rl_prof_pre(st);
  cudaLaunchKernelEx(&cfg, kernel, a, tmq, tmkv, tmp);
  return rl_check_launch("attn_fwd_umma", C, -1, rl_tf32_tag(TF32));
}

}  // namespace

// Which forward kernels serve the wide stages: 0 = the one-window mma.sync kernels of attn.cu, 2 = the tile kernels
// above, 1 (default) = the tile kernels while the launch is a single wave of CTAs (tiles * NSL <= SM count: the
// training batch of 256 windows), the one-window / two-window kernels beyond (a tile CTA is a 20 us latency chain that
// owns its SM, so throughput at large batches is better with two 16-warp CTAs per SM; measured 346 vs 276 us at
// B = 4096, C = 128).  Initialised from RALENET_ATTN_UMMA; ralenet_set_attn_umma() switches it at run time for A/B
// measurements and the agreement test.  All three compute the same function.
static int g_attn_umma = -1;
static int attn_umma_mode() {
  if (g_attn_umma < 0) {
    const char* e = getenv("RALENET_ATTN_UMMA");
    const int m = (e && *e) ? atoi(e) : RL_ATTN_UMMA_DEFAULT;
    g_attn_umma = (m < 0 || m > 2) ? RL_ATTN_UMMA_DEFAULT : m;
  }
  return g_attn_umma;
}
extern "C" int ralenet_set_attn_umma(int mode) {
  const int prev = attn_umma_mode();
  g_attn_umma = (mode < 0 || mode > 2) ? RL_ATTN_UMMA_DEFAULT : mode;
  return prev;
}

// returns 1 if the shape / batch is not handled here (caller falls through to attn_fwd_kernel)
int rl_attn_fwd_umma(const rl_attn_fwd_args* a, cudaStream_t st) {
  const int mode = attn_umma_mode();
  if (mode == 0 || a->L * a->C != 2048 || (a->C != 64 && a->C != 128)) return 1;
  if (mode == 1) {
    static int n_sm = 0;
    if (n_sm == 0) {
      int dev = 0;
      cudaGetDevice(&dev);
      if (cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n_sm <= 0) n_sm = 148;
    }
    const int ctas = (a->B * a->L + TM - 1) / TM * (a->C / CS);
    if (ctas > n_sm) return 1;
  }
  const bool tf32 = a->flags & RL_F_TF32;
  if (a->C == 128) return tf32 ? launch<128, true>(*a, st) : launch<128, false>(*a, st);
  return tf32 ? launch<64, true>(*a, st) : launch<64, false>(*a, st);
}
