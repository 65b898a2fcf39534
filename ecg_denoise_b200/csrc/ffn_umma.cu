// ffn_umma.cu -- feed-forward half for the WIDE stages (C = 64, 128) on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, accumulators in tensor memory), one CTA per (128-token tile, 128-wide hidden slice).
//
//   y = x + fc2( GELU( leconv( GELU( fc1( LN2(x) ) ) ) ) )  (+ extra)
//
// Same arithmetic as ffn.cu (reference model/transformer.py:392-395, 149-161, 54-59); modes RL_LE_NONE and
// RL_LE_PARTIAL (the convolved hidden channel 0 lives in slice 0).  Depthwise mode and 512-sample windows use ffn.cu.
//
// At the wide stages a window has only L = 32 / 16 tokens, so a tile of TM = 128 tokens = 4 / 8 whole windows forms
// the M dimension of a 128 x N UMMA.  A cluster of NSL = 4C/128 CTAs owns one token tile and SPLITS THE HIDDEN
// DIMENSION: CTA r computes hidden units [128 r, 128 r + 128) (fc1 slice -> GELU -> local enhancement -> GELU),
// multiplies by its K-slice of fc2, and the NSL partial outputs are reduced through distributed shared memory.
// Operands are staged by the CTA's threads into the canonical un-swizzled K-major core-matrix layout together
// with their tf32 remainders (umma.cuh), one elected thread issues the 3-pass split MMAs, completion is tracked
// with mbarriers (tcgen05.commit), and the epilogues read the accumulators back with tcgen05.ld.
#define RL_NT 512
#define RL_MINB 1
#include "common.cuh"
#include "umma.cuh"
#include "tma.cuh"
#include <cooperative_groups.h>

namespace cg = cooperative_groups;

RL_TRACE_DEFINE(umma)

namespace {

constexpr int TM = 128;     // tokens per tile (UMMA M)
constexpr int TS = 128;     // hidden units per CTA (UMMA N of fc1, K of fc2)
constexpr int KC = 32;      // contraction chunk staged per pipeline step
constexpr int TMEM_COLS = 256;

template <int C>
struct FwdSmem {
  static constexpr int A_FLOATS = TM * TS;             // u tile [TM][C] and later the g2 tile [TM][TS] (C <= TS)
  static constexpr int B_FLOATS = 128 * KC;            // one weight chunk (up to 128 rows)
  static constexpr size_t BYTES = sizeof(float) * (2 * A_FLOATS + 4 * B_FLOATS + 2 * TM + 2 * C) + 64;
};

using umma::Ring;

// The weight chunks of fc1 and fc2 arrive through cp.async.bulk.tensor (tma.cuh) in one 2-stage ring that runs across
// both GEMMs (chunks 0 .. C/32 - 1 from W1, then TS/32 chunks from W2); one thread issues, the CTA only derives the tf32
// remainder tile.  TF32 (RL_F_TF32): single-pass MMAs; the CTA rounds the operand tiles to tf32 instead of splitting them
// (the remainder halves of the shared-memory plan stay unused).
template <int C, bool TF32>
__global__ void __launch_bounds__(RL_NT, RL_MINB) ffn_fwd_umma_kernel(const rl_ffn_fwd_args a,
                                                                      const __grid_constant__ CUtensorMap tm1,
                                                                      const __grid_constant__ CUtensorMap tm2) {
  constexpr int L = 2048 / C, HC = 4 * C, NSL = HC / TS;
  constexpr int NCH1 = C / KC;
  extern __shared__ __align__(1024) float smem[];
  float* sA_hi = smem;
  float* sA_lo = sA_hi + FwdSmem<C>::A_FLOATS;
  float* sB = sA_lo + FwdSmem<C>::A_FLOATS;                  // [2 stages][hi | lo][128 * KC]
  float* sg10 = sB + 4 * FwdSmem<C>::B_FLOATS;               // g1[:, 0] of the tile (slice 0)
  float* sfir = sg10 + TM;
  float* s_ln = sfir + TM;                                   // norm2 weight [C] | bias [C]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_ln + 2 * C);   // [0,1]: MMAs of a ring buffer done; [2,3]: TMA landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4);
  // chunk jj of the weight ring (tid 0): fc1 rows [128 r, 128 r + 128) x K chunk jj, then fc2 rows [0, C) x its
  // K chunk inside hidden slice r
  const int r_early = blockIdx.x % NSL;
  auto tma_issue = [&](int jj) {
    const int b = jj & 1;
    float* dst = sB + b * 2 * FwdSmem<C>::B_FLOATS;
    if (jj < NCH1) {
      tma::expect_tx(bars + 2 + b, TS * KC * 4);
      tma::load_2d(dst, &tm1, jj * KC, r_early * TS, bars + 2 + b);
    } else {
      tma::expect_tx(bars + 2 + b, C * KC * 4);
      tma::load_2d(dst, &tm2, r_early * TS + (jj - NCH1) * KC, 0, bars + 2 + b);
    }
  };
  // all threads: wait for chunk jj, derive its remainder tile (same swizzled layout, element-wise; TF32: round in place)
  auto tma_consume = [&](int jj, int rows) {
    const int b = jj & 1;
    umma::mbar_wait(bars + 2 + b, (uint32_t)((jj >> 1) & 1));
    float4* hi4 = reinterpret_cast<float4*>(sB + b * 2 * FwdSmem<C>::B_FLOATS);
    float4* lo4 = reinterpret_cast<float4*>(sB + b * 2 * FwdSmem<C>::B_FLOATS + FwdSmem<C>::B_FLOATS);
    for (int i = threadIdx.x; i < rows * KC / 4; i += RL_NT) {
      const float4 v = hi4[i];
      if constexpr (TF32) hi4[i] = umma::rna4(v);
      else lo4[i] = umma::lo4(v);
    }
  };
  if (threadIdx.x == 0) {
    umma::mbar_init(bars, 1);
    umma::mbar_init(bars + 1, 1);
    umma::mbar_init(bars + 2, 1);
    umma::mbar_init(bars + 3, 1);
    umma::fence_mbar_init();
    umma::fence_async_smem();
    tma::prefetch_desc(&tm1);
    tma::prefetch_desc(&tm2);
    tma_issue(0);                        // weights are immutable inside the step: both ring buffers fill while the
    tma_issue(1);                        // previous kernel drains
  }
  // ... and so does the LayerNorm affine: staged in shared memory here, phase 1 then waits for one round of global
  // loads (x) instead of one more round per 16-byte chunk
  if ((a.flags & RL_F_PRENORM) && threadIdx.x < C / 2) {
    const int t = threadIdx.x;
    *reinterpret_cast<float4*>(s_ln + 4 * t) =
        __ldg(reinterpret_cast<const float4*>(t < C / 4 ? a.ln_w : a.ln_b) + (t % (C / 4)));
  }
  RL_TS(umma, 0);
  pdl_wait();
  pdl_trigger();
  RL_TS(umma, 1);

  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int tile = blockIdx.x / NSL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t tok0 = (size_t)tile * TM;
  const int nvalid = min(TM, a.B * L - (int)tok0);            // valid token rows of this tile
  const float* xw = a.x + tok0 * C;

  if (warp == 0) umma::tmem_alloc<TMEM_COLS>(tmem_slot);
  __syncthreads();                                           // staged LayerNorm affine visible to every warp
  RL_TS(umma, 2);

  // 1. LN2 over the TM tokens -> A tile (K-major, KT = C) with its tf32 remainder.  A warp owns 8 rows; lane =
  //    (row % 8, 16-byte chunk % 4), so global reads cover full sectors and the tile stores are contiguous.
  {
    constexpr int NI = C / 16;                                // chunks per lane
    const int rsub = lane & 7, qsub = lane >> 3;
    const int row = warp * 8 + rsub;
    const bool ok = row < nvalid;
    float4 v[NI];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      v[i] = ok ? __ldg(reinterpret_cast<const float4*>(xw + (size_t)row * C) + qsub + 4 * i)
                : make_float4(0.f, 0.f, 0.f, 0.f);
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
    float mu = 0.f, rstd = 1.f;
    if (a.flags & RL_F_PRENORM) {
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
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int qc = qsub + 4 * i;
      float4 u = v[i];
      if (a.flags & RL_F_PRENORM) {
        const float4 w4 = *reinterpret_cast<const float4*>(s_ln + 4 * qc);
        const float4 b4 = *reinterpret_cast<const float4*>(s_ln + C + 4 * qc);
        u.x = fmaf((v[i].x - mu) * rstd, w4.x, b4.x);
        u.y = fmaf((v[i].y - mu) * rstd, w4.y, b4.y);
        u.z = fmaf((v[i].z - mu) * rstd, w4.z, b4.z);
        u.w = fmaf((v[i].w - mu) * rstd, w4.w, b4.w);
        if (!ok) u = make_float4(0.f, 0.f, 0.f, 0.f);
      }
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
  RL_TS(umma, 3);

  // 2. hidden slice: h = u W1[128 r : 128 r + 128]^T   (M = TM, N = TS, K = C) -> TMEM columns [0, TS)
  {
    constexpr uint32_t idesc = umma::idesc_tf32(TM, TS);
#pragma unroll
    for (int j = 0; j < C / KC; ++j) {
      float* bh = sB + ring.buf() * 2 * FwdSmem<C>::B_FLOATS;
      float* bl = bh + FwdSmem<C>::B_FLOATS;
      tma_consume(j, TS);
      umma::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        umma::tc_fence_after();
        tma::mma_chunk_3x<KC, TF32>(tb, sA_hi, sA_lo, C, j * KC, bh, bl, idesc, j > 0 ? 1u : 0u);
        umma::commit(bars + ring.buf());
        // refill this buffer with chunk j + 2 as soon as its MMAs have drained (TS / KC >= 2: chunk j + 2 always
        // exists here)
        ++ring.chunk;
        ring.wait_last();
        --ring.chunk;
        tma_issue(j + 2);
      }
      ++ring.chunk;
    }
  }
  RL_TS(umma, 4);
  ring.wait_last();
  umma::tc_fence_after();
  RL_TS(umma, 5);

  // 3. epilogue 1: + b1, save h, GELU, local enhancement (3-tap FIR along the tokens of each window on hidden
  //    channel 0 = column 0 of slice 0), second GELU -> g2 tile (K-major, KT = TS) with remainder, over the dead u tile.
  //    warp w reads TMEM lane quadrant w % 4 (rows 32 (w % 4) ...) and the column group w / 4 (32 columns).
  {
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    const bool ok = row < nvalid;
    const int col0 = cgp * 32;                               // within the slice
    const bool part = a.le_mode == RL_LE_PARTIAL;
    float hv[32];
    {
      float t0[16], t1[16];
      umma::tmem_ld16(umma::tmem_addr(tb, col0), t0);
      umma::tmem_ld16(umma::tmem_addr(tb, col0 + 16), t1);
#pragma unroll
      for (int i = 0; i < 16; ++i) { hv[i] = t0[i]; hv[16 + i] = t1[i]; }
    }
    const float* b1 = a.b1 ? a.b1 + r * TS + col0 : nullptr;
    if (b1) {
#pragma unroll
      for (int i = 0; i < 32; i += 4) {
        const float4 b4 = __ldg(reinterpret_cast<const float4*>(b1 + i));
        hv[i] += b4.x; hv[i + 1] += b4.y; hv[i + 2] += b4.z; hv[i + 3] += b4.w;
      }
    }
    if (a.h && ok) {
      float4* hs = reinterpret_cast<float4*>(a.h + (tok0 + row) * HC + r * TS + col0);
#pragma unroll
      for (int i = 0; i < 8; ++i) hs[i] = make_float4(hv[4 * i], hv[4 * i + 1], hv[4 * i + 2], hv[4 * i + 3]);
    }
#pragma unroll
    for (int i = 0; i < 32; i += 2) gelu2(hv[i], hv[i + 1], hv[i], hv[i + 1]);
    const bool own0 = part && r == 0 && cgp == 0;            // this thread holds hidden channel 0 of its row
    if (own0) sg10[row] = hv[0];
    __syncthreads();
    if (part) {
      if (own0) {
        const int tl = row % L;
        const float w0f = __ldg(a.lew), w1f = __ldg(a.lew + 1), w2f = __ldg(a.lew + 2);
        const float p = (tl > 0) ? sg10[row - 1] : 0.f;
        const float n = (tl + 1 < L) ? sg10[row + 1] : 0.f;
        hv[0] = w0f * p + w1f * hv[0] + w2f * n;
      }
#pragma unroll
      for (int i = 0; i < 32; i += 2) gelu2(hv[i], hv[i + 1], hv[i], hv[i + 1]);
    }
    const int obase = (row & 7) * 4 + (row >> 3) * (TS / 4) * 32;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int o = obase + (col0 / 4 + i) * 32;
      const float4 g = make_float4(hv[4 * i], hv[4 * i + 1], hv[4 * i + 2], hv[4 * i + 3]);
      if constexpr (TF32) {
        *reinterpret_cast<float4*>(sA_hi + o) = umma::rna4(g);
      } else {
        *reinterpret_cast<float4*>(sA_hi + o) = g;
        *reinterpret_cast<float4*>(sA_lo + o) = umma::lo4(g);
      }
    }
  }
  umma::tc_fence_before();     // the tcgen05.ld reads of the fc1 accumulator precede the barrier below
  RL_TS(umma, 6);

  // 4. partial output of this hidden slice: yp = g2 W2[:, 128 r : 128 r + 128]^T  (M = TM, N = C, K = TS)
  //    -> TMEM columns [TS, TS + C)
  {
    constexpr uint32_t idesc = umma::idesc_tf32(TM, C);
#pragma unroll
    for (int j = 0; j < TS / KC; ++j) {
      float* bh = sB + ring.buf() * 2 * FwdSmem<C>::B_FLOATS;
      float* bl = bh + FwdSmem<C>::B_FLOATS;
      tma_consume(NCH1 + j, C);
      umma::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        umma::tc_fence_after();
        tma::mma_chunk_3x<KC, TF32>(tb + TS, sA_hi, sA_lo, TS, j * KC, bh, bl, idesc, j > 0 ? 1u : 0u);
        umma::commit(bars + ring.buf());
        if (j + 2 < TS / KC) {
          ++ring.chunk;
          ring.wait_last();
          --ring.chunk;
          tma_issue(NCH1 + j + 2);
        }
      }
      ++ring.chunk;
    }
  }
  ring.wait_last();
  umma::tc_fence_after();
  RL_TS(umma, 7);

  // 5. epilogue 2: partial tile -> shared memory [TM][C + 4] (over the dead g2 tile), DSMEM reduction:
  //    CTA r finishes rows [r * TM / NSL, (r + 1) * TM / NSL)
  constexpr int LDP = C + 4;
  float* sp = smem;
  {
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    constexpr int CW = C / 4;                                 // columns per warp group (16 or 32)
#pragma unroll
    for (int c16 = 0; c16 < CW; c16 += 16) {
      float t0[16];
      umma::tmem_ld16(umma::tmem_addr(tb, TS + cgp * CW + c16), t0);
#pragma unroll
      for (int i = 0; i < 16; i += 4)
        *reinterpret_cast<float4*>(sp + row * LDP + cgp * CW + c16 + i) = make_float4(t0[i], t0[i + 1], t0[i + 2], t0[i + 3]);
    }
  }
  umma::tc_fence_before();
  // rows [r RPC, (r + 1) RPC) are finished here: their bias + residual (+ extra) terms are fetched before the
  // cluster barrier instead of one round trip per item behind it
  constexpr int RPC = TM / NSL, RIT = RPC * (C / 4) / RL_NT;  // rows finished by this CTA, float4 items per thread
  static_assert(RPC * (C / 4) % RL_NT == 0, "reduce: items must tile the CTA");
  float4 add4[RIT];
#pragma unroll
  for (int it = 0; it < RIT; ++it) {
    const int i = tid + it * RL_NT;
    const int rr = r * RPC + i / (C / 4), c = (i % (C / 4)) * 4;
    add4[it] = a.b2 ? __ldg(reinterpret_cast<const float4*>(a.b2 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (rr < nvalid) {
      const size_t g = (tok0 + rr) * C + c;
      if (a.flags & RL_F_RESIDUAL) {
        const float4 x4 = __ldg(reinterpret_cast<const float4*>(a.x + g));
        add4[it].x += x4.x; add4[it].y += x4.y; add4[it].z += x4.z; add4[it].w += x4.w;
      }
      if (a.extra) {
        const float4 e4 = __ldg(reinterpret_cast<const float4*>(a.extra + g));
        add4[it].x += e4.x; add4[it].y += e4.y; add4[it].z += e4.z; add4[it].w += e4.w;
      }
    }
  }
  RL_TS(umma, 8);
  cluster.sync();
  RL_TS(umma, 9);
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
  RL_TS(umma, 10);
  cluster.sync();     // nobody may exit while its partial tile is still being read
  if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tb);
  RL_TS(umma, 11);
}

// ---------------------------------------------------------------------------------------------
// Backward of the same half.  Per CTA (token tile, hidden slice r):
//   dg2 = g W2[:, slice]            (UMMA, B = W2^T staged transposed)
//   dh  = dg2 through GELU' / FIR^T / GELU' (recomputed from the saved pre-activation h)   -> scratch dh, g2
//   du_partial = dh W1[slice, :]    (UMMA, B = W1^T staged transposed)
//   DSMEM reduction of the NSL partials, LayerNorm backward + residual for the rows owned by this CTA.
// The weight gradients are taken afterwards from the scratch tensors (g, g2), (dh, u) by wgrad.cu.
template <int C>
struct BwdSmem {
  static constexpr int A_FLOATS = TM * TS;
  static constexpr int B_FLOATS = 128 * KC;
  static constexpr size_t BYTES = sizeof(float) * (2 * A_FLOATS + 4 * B_FLOATS + 2 * TM + 2 * C + 64) + 64;
};

template <int C, bool DET>
__global__ void __launch_bounds__(RL_NT, RL_MINB) ffn_bwd_umma_kernel(const rl_ffn_bwd_args a) {
  constexpr int L = 2048 / C, HC = 4 * C, NSL = HC / TS;
  // dgrad operand of fc2, B(n = hidden, k = c) = W2[c][128 r + n]: prefetched before the dependency wait
  umma::TStage<TS, KC, RL_NT> w2r[C / KC];
  {
    const float* w2s = a.w2 + (size_t)(blockIdx.x % NSL) * TS;
#pragma unroll
    for (int j = 0; j < C / KC; ++j) w2r[j].load(w2s + (size_t)(j * KC) * HC, HC);
  }
  {   // the tensors the forward pass saved sit in HBM by now: pull this CTA's pre-activation slice (one 128-byte
      // line per thread: 32 hidden units of one token) and its rows of the block input towards L2
    const int tile_p = blockIdx.x / NSL, r_p = blockIdx.x % NSL;
    const long long tok = (long long)tile_p * TM + ((threadIdx.x >> 5) & 3) * 32 + (threadIdx.x & 31);
    if (tok < (long long)a.B * L) {
      prefetch_l2(a.h + tok * HC + r_p * TS + (threadIdx.x >> 7) * 32);
      if ((int)(threadIdx.x >> 7) < C / 32) prefetch_l2(a.x + tok * C + (threadIdx.x >> 7) * 32);
    }
  }
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(1024) float smem[];
  float* sA_hi = smem;
  float* sA_lo = sA_hi + BwdSmem<C>::A_FLOATS;
  float* sB = sA_lo + BwdSmem<C>::A_FLOATS;
  float* sg10 = sB + 4 * BwdSmem<C>::B_FLOATS;               // g1[:, 0]   (slice 0)
  float* sdf0 = sg10 + TM;                                   // df[:, 0]
  float* s_gb = sdf0 + TM;                                   // LayerNorm weight / bias gradient partials
  float* s_red = s_gb + 2 * C;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_red + 64);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);

  cg::cluster_group cluster = cg::this_cluster();
  const int r = (int)cluster.block_rank();
  const int tile = blockIdx.x / NSL;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const size_t tok0 = (size_t)tile * TM;
  const int nvalid = min(TM, a.B * L - (int)tok0);
  const float* gw = a.g + tok0 * C;
  const int mode = a.le_mode;
  const bool part0 = (mode == RL_LE_PARTIAL) && (r == 0);

  if (tid == 0) {
    umma::mbar_init(bars, 1);
    umma::mbar_init(bars + 1, 1);
    umma::fence_mbar_init();
  }
  if (warp == 0) umma::tmem_alloc<TMEM_COLS>(tmem_slot);

  // 1. g tile -> A (K-major, KT = C) with remainder
  {
    constexpr int NI = C / 16;
    const int rsub = lane & 7, qsub = lane >> 3;
    const int row = warp * 8 + rsub;
    const bool ok = row < nvalid;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const int qc = qsub + 4 * i;
      const float4 v = ok ? __ldg(reinterpret_cast<const float4*>(gw + (size_t)row * C) + qc)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
      const int o = rsub * 4 + qc * 32 + warp * (C / 4) * 32;
      *reinterpret_cast<float4*>(sA_hi + o) = v;
      *reinterpret_cast<float4*>(sA_lo + o) = umma::lo4(v);
    }
  }
  umma::tc_fence_before();
  __syncthreads();
  umma::tc_fence_after();
  const uint32_t tb = *tmem_slot;
  Ring ring{bars, 0};

  // 2. dg2 slice = g W2[:, slice]   (M = TM, N = TS, K = C) -> TMEM columns [0, TS)
  {
    constexpr uint32_t idesc = umma::idesc_tf32(TM, TS);
#pragma unroll
    for (int j = 0; j < C / KC; ++j) {
      ring.wait_free();
      float* bh = sB + ring.buf() * 2 * BwdSmem<C>::B_FLOATS;
      float* bl = bh + BwdSmem<C>::B_FLOATS;
      w2r[j].store(bh, bl);
      umma::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        umma::tc_fence_after();
        umma::mma_chunk_3x<KC>(tb, sA_hi, sA_lo, C, j * KC, bh, bl, idesc, j > 0 ? 1u : 0u);
        umma::commit(bars + ring.buf());
      }
      ++ring.chunk;
    }
  }
  // dgrad operand of fc1, B(n = c, k = hidden) = W1[128 r + k][n]: in flight during the epilogue below
  umma::TStage<C, KC, RL_NT> w1r[TS / KC];
  {
    const float* w1s = a.w1 + (size_t)r * TS * C;
#pragma unroll
    for (int j = 0; j < TS / KC; ++j) w1r[j].load(w1s + (size_t)(j * KC) * C, C);
  }

  // 3. epilogue 1: dg2 -> dh through GELU' / FIR^T / GELU'; g2 and dh go to the scratch tensors of the weight
  //    gradients, dh also becomes the A tile (K-major, KT = TS) of the second GEMM (over the dead g tile)
  {
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    const bool ok = row < nvalid;
    const int col0 = cgp * 32;
    const size_t hoff = (tok0 + row) * HC + r * TS + col0;
    const bool own0 = part0 && cgp == 0;                     // this thread holds hidden channel 0 of its row
    float lw0 = 0.f, lw1 = 0.f, lw2 = 0.f, h0 = 0.f, g10 = 0.f, f0 = 0.f;
    if (part0) { lw0 = __ldg(a.lew); lw1 = __ldg(a.lew + 1); lw2 = __ldg(a.lew + 2); }
    if (own0) {
      h0 = ok ? __ldg(a.h + hoff) : 0.f;
      g10 = gelu_f(h0);
      sg10[row] = g10;
    }
    __syncthreads();
    if (own0) {
      const int tl = row % L;
      const float p = (tl > 0) ? sg10[row - 1] : 0.f;
      const float n = (tl + 1 < L) ? sg10[row + 1] : 0.f;
      f0 = lw0 * p + lw1 * g10 + lw2 * n;
    }
    ring.wait_last();
    umma::tc_fence_after();
    const int obase = (row & 7) * 4 + (row >> 3) * (TS / 4) * 32;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      float v[16], hh[16], g2v[16];
      umma::tmem_ld16(umma::tmem_addr(tb, col0 + 16 * half), v);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float4 t4 = ok ? __ldg(reinterpret_cast<const float4*>(a.h + hoff + 16 * half) + i)
                             : make_float4(0.f, 0.f, 0.f, 0.f);
        hh[4 * i] = t4.x; hh[4 * i + 1] = t4.y; hh[4 * i + 2] = t4.z; hh[4 * i + 3] = t4.w;
      }
#pragma unroll
      for (int i = 0; i < 16; i += 2) {                      // two hidden units at a time on the packed fp32 pipe
        float g1[2], d1[2];
        gelu_both2(hh[i], hh[i + 1], g1[0], g1[1], d1[0], d1[1]);
        if (mode == RL_LE_NONE) {
          g2v[i] = g1[0]; g2v[i + 1] = g1[1];
          v[i] *= d1[0]; v[i + 1] *= d1[1];
        } else {
          // second GELU: the convolved channel (column 0 of slice 0) takes the FIR output, the others f == g1
          const bool conv0 = own0 && half == 0 && i == 0;
          float g2[2], d2[2];
          gelu_both2(conv0 ? f0 : g1[0], g1[1], g2[0], g2[1], d2[0], d2[1]);
          g2v[i] = g2[0]; g2v[i + 1] = g2[1];
          if (conv0) {                                       // finished after the FIR adjoint
            sdf0[row] = v[i] * d2[0];
            v[i] = 0.f;
          } else {
            v[i] *= d2[0] * d1[0];
          }
          v[i + 1] *= d2[1] * d1[1];
        }
      }
      if (ok) {
        float4* g2p = reinterpret_cast<float4*>(a.g2 + hoff + 16 * half);
        float4* dhp = reinterpret_cast<float4*>(a.dh + hoff + 16 * half);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          g2p[i] = make_float4(g2v[4 * i], g2v[4 * i + 1], g2v[4 * i + 2], g2v[4 * i + 3]);
          dhp[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int o = obase + (col0 / 4 + 4 * half + i) * 32;
        const float4 d = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        *reinterpret_cast<float4*>(sA_hi + o) = d;
        *reinterpret_cast<float4*>(sA_lo + o) = umma::lo4(d);
      }
    }
    __syncthreads();
    if (part0) {                                             // adjoint of the 3-tap FIR on hidden channel 0
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      if (own0) {
        const int tl = row % L;
        const float d = sdf0[row];
        const float dn = (tl + 1 < L) ? sdf0[row + 1] : 0.f;
        const float dp = (tl > 0) ? sdf0[row - 1] : 0.f;
        const float dg1 = lw0 * dn + lw1 * d + lw2 * dp;
        const float dh = ok ? dg1 * gelu_grad_f(h0) : 0.f;
        if (ok) a.dh[hoff] = dh;
        const int o = obase + (col0 / 4) * 32;               // element (row, k = 0) of the dh tile
        sA_hi[o] = dh;
        sA_lo[o] = dh - umma::trunc_tf32(dh);
        a0 = d * ((tl > 0) ? sg10[row - 1] : 0.f);
        a1 = d * g10;
        a2 = d * ((tl + 1 < L) ? sg10[row + 1] : 0.f);
      }
      if (a.d_lew) {
        a0 = block_sum(a0, s_red);
        a1 = block_sum(a1, s_red);
        a2 = block_sum(a2, s_red);
        if (tid == 0) {
          float* d_lew = grad_slot<DET>(a.d_lew, 3, tile);   // one slot per token tile (its rank-0 CTA)
          grad_add<DET>(d_lew, a0);
          grad_add<DET>(d_lew + 1, a1);
          grad_add<DET>(d_lew + 2, a2);
        }
      }
    }
  }
  umma::tc_fence_before();

  // 4. partial du = dh_slice W1[slice rows, :]   (M = TM, N = C, K = TS) -> TMEM columns [TS, TS + C)
  {
    constexpr uint32_t idesc = umma::idesc_tf32(TM, C);
#pragma unroll
    for (int j = 0; j < TS / KC; ++j) {
      ring.wait_free();
      float* bh = sB + ring.buf() * 2 * BwdSmem<C>::B_FLOATS;
      float* bl = bh + BwdSmem<C>::B_FLOATS;
      w1r[j].store(bh, bl);
      umma::fence_async_smem();
      __syncthreads();
      if (tid == 0) {
        umma::tc_fence_after();
        umma::mma_chunk_3x<KC>(tb + TS, sA_hi, sA_lo, TS, j * KC, bh, bl, idesc, j > 0 ? 1u : 0u);
        umma::commit(bars + ring.buf());
      }
      ++ring.chunk;
    }
  }
  ring.wait_last();
  umma::tc_fence_after();

  // 5. partial tile -> shared memory, DSMEM reduction + LayerNorm backward: CTA r finishes rows [r RPC, (r+1) RPC)
  constexpr int LDP = C + 4;
  float* sp = smem;
  {
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    constexpr int CW = C / 4;
#pragma unroll
    for (int c16 = 0; c16 < CW; c16 += 16) {
      float t0[16];
      umma::tmem_ld16(umma::tmem_addr(tb, TS + cgp * CW + c16), t0);
#pragma unroll
      for (int i = 0; i < 16; i += 4)
        *reinterpret_cast<float4*>(sp + row * LDP + cgp * CW + c16 + i) = make_float4(t0[i], t0[i + 1], t0[i + 2], t0[i + 3]);
    }
  }
  umma::tc_fence_before();
  cluster.sync();
  {
    constexpr int RPC = TM / NSL;
    const float* part[NSL];
#pragma unroll
    for (int q = 0; q < NSL; ++q) part[q] = cluster.map_shared_rank(sp, q);
    const int row0 = r * RPC;
    const int rows_here = max(0, min(RPC, nvalid - row0));
    float* dxw = a.dx + (tok0 + row0) * C;
    float* uw = a.u + (tok0 + row0) * C;
    const float* xr = a.x + (tok0 + row0) * C;
    const float* gr = gw + (size_t)row0 * C;
    const bool resid = a.flags & RL_F_RESIDUAL;
    auto du_at4 = [&](int t, int c) {          // four channels of the reduced partial tiles (16-byte DSMEM loads)
      const int off = (row0 + t) * LDP + c;
      float4 s = *reinterpret_cast<const float4*>(part[0] + off);
#pragma unroll
      for (int q = 1; q < NSL; ++q) {
        const float4 p = *reinterpret_cast<const float4*>(part[q] + off);
        s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
      }
      return s;
    };
    if (a.flags & RL_F_PRENORM) {
      const float* lw = a.ln_w;
      const float* lb = a.ln_b;
      // per-warp partial rows of the LayerNorm weight / bias gradients: the weight ring (dead by now), 16 x 2C floats
      static_assert(32 * C <= 4 * BwdSmem<C>::B_FLOATS, "ffn_bwd_umma: partial rows");
      ln_backward_rows4<C, true>(
          rows_here, lw, sB, [&](int t, int c) { return ldg4(xr + t * C + c); }, du_at4,
          [&](int t, int c, float4 dz, float4 zh) {
            if (resid) {
              const float4 g4 = ldg4(gr + t * C + c);
              dz.x += g4.x; dz.y += g4.y; dz.z += g4.z; dz.w += g4.w;
            }
            *reinterpret_cast<float4*>(dxw + t * C + c) = dz;
            *reinterpret_cast<float4*>(uw + t * C + c) = fma4(zh, ldg4(lw + c), ldg4(lb + c));
          });
      __syncthreads();
      ln_backward_finish<C, DET>(sB, grad_slot<DET>(a.d_ln_w, C, blockIdx.x), grad_slot<DET>(a.d_ln_b, C, blockIdx.x));
    } else {
      for (int i = tid; i < rows_here * C / 4; i += RL_NT) {
        const int t = (4 * i) / C, c = (4 * i) % C;
        float4 d = du_at4(t, c);
        if (resid) {
          const float4 g4 = ldg4(gr + 4 * i);
          d.x += g4.x; d.y += g4.y; d.z += g4.z; d.w += g4.w;
        }
        *reinterpret_cast<float4*>(dxw + 4 * i) = d;
        *reinterpret_cast<float4*>(uw + 4 * i) = ldg4(xr + 4 * i);
      }
    }
  }
  cluster.sync();
  if (warp == 0) umma::tmem_dealloc<TMEM_COLS>(tb);
}

template <typename Args>
int launch_cluster(void (*kernel)(const Args), size_t smem, int grid, int cl, const Args& a, cudaStream_t st,
                   const char* name, int C) {
  if (int rc = rl_set_smem(kernel, smem)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(RL_NT);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cl;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  rl_prof_pre(st);
  cudaLaunchKernelEx(&cfg, kernel, a);
  return rl_check_launch(name, C);
}

}  // namespace

template <int C, bool TF32>
static int launch_fwd(const rl_ffn_fwd_args* a, int tiles, cudaStream_t st) {
  constexpr int NSL = 4 * C / TS;
  CUtensorMap tm1 = {}, tm2 = {};
  if (int rc = rl_tmap_weight(a->w1, 4 * C, C, C, TS, &tm1)) return rc;           // fc1 [4C][C]: 128-row slices
  if (int rc = rl_tmap_weight(a->w2, C, 4 * C, 4 * C, C, &tm2)) return rc;        // fc2 [C][4C]: all C rows
  auto kernel = ffn_fwd_umma_kernel<C, TF32>;
  const size_t smem = FwdSmem<C>::BYTES + 64;
  if (int rc = rl_set_smem(kernel, smem)) return rc;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(tiles * NSL);
  cfg.blockDim = dim3(RL_NT);
  cfg.dynamicSmemBytes = smem;
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
  cudaLaunchKernelEx(&cfg, kernel, *a, tm1, tm2);
  return rl_check_launch("ffn_fwd_umma", C, -1, rl_tf32_tag(TF32));
}

// returns 1 if the shape/mode is not handled here (caller falls through to the per-window kernels in ffn.cu)
int rl_ffn_fwd_umma(const rl_ffn_fwd_args* a, cudaStream_t st) {
  if (a->L * a->C != 2048 || a->le_mode == RL_LE_DEPTHWISE) return 1;
  const int tiles = (a->B * a->L + TM - 1) / TM;
  const bool tf32 = a->flags & RL_F_TF32;
  if (a->C == 128) return tf32 ? launch_fwd<128, true>(a, tiles, st) : launch_fwd<128, false>(a, tiles, st);
  if (a->C == 64) return tf32 ? launch_fwd<64, true>(a, tiles, st) : launch_fwd<64, false>(a, tiles, st);
  return 1;
}

template <int C>
static int launch_bwd(const rl_ffn_bwd_args* a, int tiles, cudaStream_t st, RlDet* det) {
  constexpr int NSL = 4 * C / TS;
  if (det == nullptr)
    return launch_cluster(ffn_bwd_umma_kernel<C, false>, BwdSmem<C>::BYTES, tiles * NSL, NSL, *a, st, "ffn_bwd_umma", C);
  // det: LayerNorm partials one slot per CTA, local-enhancement taps one slot per token tile
  rl_ffn_bwd_args d = *a;
  d.d_ln_w = rl_det_take(det, a->d_ln_w, C, tiles * NSL);
  d.d_ln_b = rl_det_take(det, a->d_ln_b, C, tiles * NSL);
  d.d_lew = (a->le_mode == RL_LE_PARTIAL) ? rl_det_take(det, a->d_lew, 3, tiles) : nullptr;
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "ffn_bwd: deterministic-mode workspace too small");
  return launch_cluster(ffn_bwd_umma_kernel<C, true>, BwdSmem<C>::BYTES, tiles * NSL, NSL, d, st, "ffn_bwd_umma", C);
}

int rl_ffn_bwd_umma(const rl_ffn_bwd_args* a, cudaStream_t st, RlDet* det) {
  if (a->L * a->C != 2048 || a->le_mode == RL_LE_DEPTHWISE) return 1;
  const int tiles = (a->B * a->L + TM - 1) / TM;
  if (a->C == 128) return launch_bwd<128>(a, tiles, st, det);
  if (a->C == 64) return launch_bwd<64>(a, tiles, st, det);
  return 1;
}
