// wgrad_reg.cu -- weight-gradient GEMMs over the token dimension with REGISTER-resident tiles, operands streamed
// straight from global memory into tensor-core fragments (no shared-memory staging, no transposes).
//
//   dW[n][k] += sum_t dY[t][n] X[t][k],   db[n] += sum_t dY[t][n]        (all weight matrices of one half-block)
//
// This is a tall-skinny reduction: N, K <= 512 but t runs over every token of the batch (65,536 ... 1,048,576), so
// the arithmetic intensity is 2NK / (4 (N + K)) = 8 ... 50 FLOP/B -- left of the ridge: the roof is HBM, and both
// operands should cross it exactly once.  The token-major layout of the operands IS the fragment layout of
// mma.sync.m16n8k8 when the token axis is the contraction axis:
//   A (16 x 8, rows = n, cols = tokens):  a0/a1 = dY[t0 + t][n..], a2/a3 = dY[t0 + t + 4][n..]
//   B ( 8 x 8, rows = tokens, cols = k):  b0    = X [t0 + t][k..], b1    = X [t0 + t + 4][k..]      (lane = 4 g + t)
// One 16-byte load per lane and token row covers 32 consecutive channels over the 8 g-lanes (a full 128-byte line);
// its four components feed four different MMA tiles (rows / columns are assigned to tiles as n0 + 4 g + j), so a
// warp tile of 32 x 32 outputs costs 4 LDG.128 per 8 tokens, 32 split operations (3xTF32, fp32-grade) and 24 MMAs.
// The accumulators never leave registers until the warp's token range is exhausted; the token sub-ranges of a CTA
// are then summed in shared memory and added to dW with 16-byte vector reductions.
// Measured against the tcgen05 kernels of wgrad_umma.cu (which spend their time transposing token chunks into
// K-major shared-memory tiles and splitting them there): see DESIGN.md section 4.
#define RL_NT 256
#include "common.cuh"

namespace {

constexpr int WT = 32;                      // warp tile: WT x WT outputs
constexpr int NW = RL_NT / 32;

struct RgProblem {
  const float* dY; const float* X; float* dW; float* db;
  int ldy, ldx, N, K;
  int tiles_k;        // K / 32
  int ntiles;         // (N / 32) * (K / 32)
  int cta_begin;      // first CTA column of this problem
};
struct RgGroup {
  RgProblem p[4];
  int nprob, M, MC;   // tokens, tokens per CTA slice
  int tpc;            // warp tiles per CTA (1, 2, 4, 8); NW / tpc token sub-ranges per CTA
};

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void red_add_v4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}

template <bool DET>
__global__ void __launch_bounds__(RL_NT, 2) wgrad_reg_kernel(const RgGroup grp) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();
  __shared__ __align__(16) float s_acc[NW][WT * (WT + 4)];     // one 32 x 32 tile per warp (row stride 36: no conflicts)
  __shared__ float s_bias[NW][WT];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  int pi = 0;
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (i < grp.nprob && (int)blockIdx.x >= grp.p[i].cta_begin) pi = i;
  const RgProblem& P = grp.p[pi];
  const int tpc = grp.tpc, nts = NW / tpc;
  const int tile = ((int)blockIdx.x - P.cta_begin) * tpc + warp % tpc;      // warp tile of this warp
  const int tsub = warp / tpc;
  const bool live = tile < P.ntiles;
  const int n0 = (tile / P.tiles_k) * WT, k0 = (tile % P.tiles_k) * WT;
  const int m_begin = blockIdx.y * grp.MC, m_end = min(grp.M, m_begin + grp.MC);
  const bool do_bias = live && P.db != nullptr && k0 == 0;

  float acc[2][4][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.f;
  float4 bsum = make_float4(0.f, 0.f, 0.f, 0.f);

  if (live) {
    const float* pa = P.dY + n0 + 4 * g;
    const float* pb = P.X + k0 + 4 * g;
    const size_t ldy = P.ldy, ldx = P.ldx;
    const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto load = [&](int t0, float4& a_lo4, float4& a_hi4, float4& b_lo4, float4& b_hi4) {
      const int r0 = t0 + t, r1 = t0 + t + 4;
      a_lo4 = r0 < m_end ? ldg4(pa + (size_t)r0 * ldy) : z4;
      b_lo4 = r0 < m_end ? ldg4(pb + (size_t)r0 * ldx) : z4;
      a_hi4 = r1 < m_end ? ldg4(pa + (size_t)r1 * ldy) : z4;
      b_hi4 = r1 < m_end ? ldg4(pb + (size_t)r1 * ldx) : z4;
    };
    const int step = 8 * nts;
    int t0 = m_begin + 8 * tsub;
    float4 a0v, a1v, b0v, b1v;                  // token rows t0 + t and t0 + t + 4
    if (t0 < m_end) load(t0, a0v, a1v, b0v, b1v);
    for (; t0 < m_end; t0 += step) {
      float4 na0 = z4, na1 = z4, nb0 = z4, nb1 = z4;
      if (t0 + step < m_end) load(t0 + step, na0, na1, nb0, nb1);      // next step's lines are in flight during the MMAs
      if (do_bias) {
        bsum.x += a0v.x + a1v.x; bsum.y += a0v.y + a1v.y; bsum.z += a0v.z + a1v.z; bsum.w += a0v.w + a1v.w;
      }
      // component c of the A loads: output row n0 + 4 g + c.  m16 tile i holds rows (4 g + 2 i) and (4 g + 2 i + 1)
      // as its fragment rows g and g + 8.
      const float av0[4] = {a0v.x, a0v.y, a0v.z, a0v.w}, av1[4] = {a1v.x, a1v.y, a1v.z, a1v.w};
      const float bv0[4] = {b0v.x, b0v.y, b0v.z, b0v.w}, bv1[4] = {b1v.x, b1v.y, b1v.z, b1v.w};
      uint32_t ahi[2][4], alo[2][4], bhi[4][2], blo[4][2];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        split_tf32x2(av0[2 * i], av0[2 * i + 1], ahi[i][0], ahi[i][1], alo[i][0], alo[i][1]);
        split_tf32x2(av1[2 * i], av1[2 * i + 1], ahi[i][2], ahi[i][3], alo[i][2], alo[i][3]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {             // n8 tile j holds output column k0 + 4 g + j as its fragment column g
        split_tf32x2(bv0[j], bv1[j], bhi[j][0], bhi[j][1], blo[j][0], blo[j][1]);
      }
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          mma_tf32(acc[i][j], alo[i], bhi[j]);
          mma_tf32(acc[i][j], ahi[i], blo[j]);
          mma_tf32(acc[i][j], ahi[i], bhi[j]);
        }
      a0v = na0; a1v = na1; b0v = nb0; b1v = nb1;
    }
  }

  // accumulator fragment (i, j): c0 = (row g, col 2t), c1 = (g, 2t+1), c2 = (g+8, 2t), c3 = (g+8, 2t+1) of tile (i, j);
  // tile row r -> output row 4 (r % 8) + 2 i + r / 8, tile column c -> output column 4 c + j
  float* sa = s_acc[warp];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int row = 4 * g + 2 * i + (e >> 1), col = 4 * (2 * t + (e & 1)) + j;
        sa[row * (WT + 4) + col] = acc[i][j][e];
      }
  if (do_bias) {
    // lanes with the same g hold the same four rows for different token rows: fold the 4 t-lanes
    bsum.x += __shfl_xor_sync(0xffffffffu, bsum.x, 1); bsum.x += __shfl_xor_sync(0xffffffffu, bsum.x, 2);
    bsum.y += __shfl_xor_sync(0xffffffffu, bsum.y, 1); bsum.y += __shfl_xor_sync(0xffffffffu, bsum.y, 2);
    bsum.z += __shfl_xor_sync(0xffffffffu, bsum.z, 1); bsum.z += __shfl_xor_sync(0xffffffffu, bsum.z, 2);
    bsum.w += __shfl_xor_sync(0xffffffffu, bsum.w, 1); bsum.w += __shfl_xor_sync(0xffffffffu, bsum.w, 2);
    if (t == 0) {
      s_bias[warp][4 * g] = bsum.x; s_bias[warp][4 * g + 1] = bsum.y;
      s_bias[warp][4 * g + 2] = bsum.z; s_bias[warp][4 * g + 3] = bsum.w;
    }
  }
  __syncthreads();
  // sum the token sub-ranges of every warp tile of this CTA and add the tile to dW: 256 float4 per tile
  for (int it = tid; it < tpc * (WT * WT / 4); it += RL_NT) {
    const int wt = it / (WT * WT / 4), q = it % (WT * WT / 4), row = q / (WT / 4), c4 = (q % (WT / 4)) * 4;
    const int tl = ((int)blockIdx.x - P.cta_begin) * tpc + wt;
    if (tl >= P.ntiles) continue;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int ts = 0; ts < nts; ++ts) {
      const float4 v = *reinterpret_cast<const float4*>(&s_acc[ts * tpc + wt][row * (WT + 4) + c4]);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    const int nn = (tl / P.tiles_k) * WT + row, kk = (tl % P.tiles_k) * WT + c4;
    if constexpr (DET)      // slot = token slice blockIdx.y of the partial slab
      *reinterpret_cast<float4*>(grad_slot<DET>(P.dW, (size_t)P.N * P.K, blockIdx.y) + (size_t)nn * P.K + kk) = s;
    else
      red_add_v4(P.dW + (size_t)nn * P.K + kk, s);
  }
  if (P.db != nullptr)
    for (int it = tid; it < tpc * WT; it += RL_NT) {
      const int wt = it / WT, row = it % WT;
      const int tl = ((int)blockIdx.x - P.cta_begin) * tpc + wt;
      if (tl >= P.ntiles || tl % P.tiles_k != 0) continue;
      float s = 0.f;
      for (int ts = 0; ts < nts; ++ts) s += s_bias[ts * tpc + wt][row];
      grad_add<DET>(grad_slot<DET>(P.db, P.N, blockIdx.y) + (tl / P.tiles_k) * WT + row, s);
    }
}

int g_wgrad_reg = -1;
int wgrad_reg_on() {
  if (g_wgrad_reg < 0) {
    const char* e = getenv("RALENET_WGRAD_REG");
    g_wgrad_reg = (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1;
  }
  return g_wgrad_reg;
}

}  // namespace

extern "C" int ralenet_set_wgrad_reg(int on) {
  const int prev = wgrad_reg_on();
  g_wgrad_reg = on < 0 ? 0 : (on > 2 ? 2 : on);      // 2: also the large groups (tests, A/B)
  return prev;
}

// returns 1 when the group is not handled here (caller falls through to wgrad_umma.cu / wgrad.cu)
int rl_launch_wgrad_group_reg(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det) {
  if (!wgrad_reg_on() || M < 64) return 1;
  RgGroup grp;
  grp.nprob = 0;
  grp.M = M;
  int max_tiles = 0;
  for (int i = 0; i < n; ++i) {
    if (!d[i].dW) continue;
    if (grp.nprob == 4) return 1;
    if (d[i].N % WT || d[i].K % WT || d[i].ldy % 4 || d[i].ldx % 4 || (uintptr_t)d[i].dY % 16 || (uintptr_t)d[i].X % 16 ||
        (uintptr_t)d[i].dW % 16)
      return 1;
    RgProblem& p = grp.p[grp.nprob++];
    p.dY = d[i].dY; p.X = d[i].X; p.dW = d[i].dW; p.db = d[i].db;
    p.ldy = d[i].ldy; p.ldx = d[i].ldx; p.N = d[i].N; p.K = d[i].K;
    p.tiles_k = p.K / WT;
    p.ntiles = (p.N / WT) * p.tiles_k;
    max_tiles = max(max_tiles, p.ntiles);
  }
  if (grp.nprob == 0) return RL_OK;
  // Large dW (more than four 32 x 32 tiles: the C >= 64 stages) are bound by the 3-pass mma.sync tensor rate, where the
  // tcgen05 kernels of wgrad_umma.cu are 2.4x faster (measured: C = 128 feed-forward pair 364 vs 233 us at 65,536
  // tokens); this kernel takes the HBM-bound small ones (C = 32 attention group 81 vs 298 us at 262,144 tokens).
  if (max_tiles > 4 && wgrad_reg_on() != 2) return 1;
  // warp tiles per CTA: consecutive tiles of a CTA share their dY rows (L1 hits); the remaining warps split the tokens
  grp.tpc = max_tiles >= 8 ? 8 : (max_tiles >= 4 ? 4 : (max_tiles >= 2 ? 2 : 1));
  int ctas = 0;
  for (int i = 0; i < grp.nprob; ++i) {
    grp.p[i].cta_begin = ctas;
    ctas += (grp.p[i].ntiles + grp.tpc - 1) / grp.tpc;
  }
  for (int i = grp.nprob; i < 4; ++i) grp.p[i] = grp.p[0];
  // token slices: two waves of 2 CTAs per SM at most, never shorter than 64 tokens per token sub-range
  const int nts = NW / grp.tpc;
  int splits = (2 * 2 * 148 + ctas - 1) / ctas;
  const int max_splits = max(1, M / (64 * nts));
  splits = max(1, min(splits, max_splits));
  if (det) splits = min(splits, RL_DET_MAX_SPLIT);
  int MC = (M + splits - 1) / splits;
  MC = (MC + 8 * nts - 1) / (8 * nts) * (8 * nts);
  splits = (M + MC - 1) / MC;
  grp.MC = MC;
  if (det == nullptr) {
    rl_launch_pdl(wgrad_reg_kernel<false>, dim3(ctas, splits), dim3(RL_NT), 0, st, grp);
    return rl_check_launch("wgrad_reg_kernel", max_tiles, ctas);
  }
  for (int i = 0; i < grp.nprob; ++i) {     // one partial slot per token slice
    RgProblem& p = grp.p[i];
    p.dW = rl_det_take(det, p.dW, (size_t)p.N * p.K, splits);
    p.db = rl_det_take(det, p.db, p.N, splits);
  }
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "wgrad: deterministic-mode workspace too small");
  for (int i = grp.nprob; i < 4; ++i) grp.p[i] = grp.p[0];
  rl_launch_pdl(wgrad_reg_kernel<true>, dim3(ctas, splits), dim3(RL_NT), 0, st, grp);
  return rl_check_launch("wgrad_reg_kernel", max_tiles, ctas);
}
