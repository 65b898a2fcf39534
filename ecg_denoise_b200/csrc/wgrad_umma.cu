// wgrad_umma.cu -- weight-gradient GEMMs over the token dimension on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, 3-pass split, accumulator in tensor memory), split over the tokens across CTAs.
//
//   dW[n][k] += sum_m dY[m][n] X[m][k]        db[n] += sum_m dY[m][n]        m = all B*L tokens of the batch
//
// These GEMMs are a third of the FLOPs of a training step.  They run on a side stream next to the data-gradient
// chain (net.cu), so their cost is what they take from the chain's SMs: the mma.sync version (wgrad.cu: 64 x 64
// tiles, 444 CTAs) cost the step 0.30 ms of its 2.33 ms.  Here a CTA owns a 128 x TK tile of one dW (or of its
// transpose, when dW has fewer than 128 rows but >= 128 columns) and a slice of tokens:
//   * both operands are token-major in global memory ([m][n], [m][k]) while the MMA wants the contraction (token)
//     index contiguous: chunks of KC = 32 tokens are transposed on the way to shared memory (32 consecutive n of four
//     consecutive tokens per warp load, one 16-byte K-major chunk per lane) together with their tf32 remainders;
//   * 2-stage shared-memory ring, and the global loads of chunks j + 1 and j + 2 are in flight (registers) while
//     chunk j is staged and its MMAs issued;
//   * epilogue: TMEM -> registers -> fp32 red.global into dW, as 16-byte vector reductions along a row (scalar ones,
//     one row per lane, are 32 L2 sector operations per warp instruction and took half of the kernel); the bias
//     gradient is summed from the staged registers of the dY operand.
// Up to 4 problems that share the token dimension and the tile width go into one launch (all weight matrices of a
// half-block).  Shapes this kernel does not take (columns not a multiple of 32, tiny M) stay on wgrad.cu.
#define RL_NT 512
#define RL_MINB 1
#include "common.cuh"
#include "umma.cuh"
#include <stdlib.h>

#ifndef RL_WGRAD_UMMA_DEFAULT
#define RL_WGRAD_UMMA_DEFAULT 1
#endif

namespace {

constexpr int TN = 128;          // rows of the output tile (UMMA M)
constexpr int KC = 32;           // tokens per chunk (contraction)
using umma::Ring;

struct WuProblem {
  const float* a;  int lda;      // row operand:    out row r    <- a[m * lda + r]
  const float* b;  int ldb;      // column operand: out column c <- b[m * ldb + c]
  float* out; int so_r, so_c;    // out[r * so_r + c * so_c] += ...
  float* bias_a;                 // += sum_m a[m][r]   (dY is the row operand)    or NULL
  float* bias_b;                 // += sum_m b[m][c]   (dY is the column operand) or NULL
  int rows, tiles_c, tile_begin; // valid rows of the problem, column tiles, first tile (blockIdx.x) of the problem
};
struct WuGroup {
  WuProblem p[4];
  int nprob, M, MC;
};

// one chunk of an operand: ROWS output rows (or columns) x KC tokens, transposed into a K-major tile pair.
// A warp reads 32 consecutive rows of four consecutive tokens and each lane owns one 16-byte chunk (its row, four
// tokens) of the tile (umma::TStage with row / token guards).
template <int ROWS>
struct TokStage {
  static constexpr int NB = ROWS / 32, NQ = KC / 4, ITEMS = NB * NQ, NWARP = RL_NT / 32;
  static constexpr int PER = (ITEMS + NWARP - 1) / NWARP;
  static_assert(ROWS % 32 == 0, "TokStage: tile shape");
  float4 v[PER];

  // src -> first row of the tile at token m0; rows_valid rows, tokens [m0, m_end) exist
  __device__ __forceinline__ void load(const float* __restrict__ src, int ld, int rows_valid, int m0, int m_end) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int item = wid + i * NWARP;
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (item < ITEMS) {
        const int nb = item % NB, q = item / NB;
        const int n = nb * 32 + lane, m = m0 + 4 * q;
        if (n < rows_valid) {
          const float* p = src + (size_t)m * ld + n;
          if (m + 3 < m_end) {
            v[i] = make_float4(__ldg(p), __ldg(p + ld), __ldg(p + 2 * (size_t)ld), __ldg(p + 3 * (size_t)ld));
          } else {
            if (m < m_end) v[i].x = __ldg(p);
            if (m + 1 < m_end) v[i].y = __ldg(p + ld);
            if (m + 2 < m_end) v[i].z = __ldg(p + 2 * (size_t)ld);
          }
        }
      }
    }
  }
  __device__ __forceinline__ void store(float* hi, float* lo) const {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int item = wid + i * NWARP;
      if (item < ITEMS) {
        const int nb = item % NB, q = item / NB;
        const int n = nb * 32 + lane;
        const int o = (n & 7) * 4 + q * 32 + (n >> 3) * (NQ * 32);
        *reinterpret_cast<float4*>(hi + o) = v[i];
        *reinterpret_cast<float4*>(lo + o) =
            umma::lo4(v[i]);
      }
    }
  }
  // sum over the staged tokens of the row this thread holds (every item of a thread has the same row:
  // NWARP % NB == 0)
  __device__ __forceinline__ float token_sum() const {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    return s;
  }
  __device__ __forceinline__ int my_row() const { return ((threadIdx.x >> 5) % NB) * 32 + (threadIdx.x & 31); }
  __device__ __forceinline__ bool active() const { return (int)(threadIdx.x >> 5) < ITEMS; }
};

template <int TK>
struct WuSmem {
  static constexpr int STAGE = 2 * TN * KC + 2 * TK * KC;     // A hi | A lo | B hi | B lo
  static constexpr size_t BYTES = sizeof(float) * (2 * STAGE + TN + TK) + 64;
};

template <int TK, bool DET>
__global__ void __launch_bounds__(RL_NT, RL_MINB) wgrad_umma_kernel(const WuGroup grp) {
  constexpr int TCOLS = (TK < 32) ? 32 : TK;                  // TMEM columns (power of two >= 32)
  static_assert((RL_NT / 32) % (TN / 32) == 0 && (RL_NT / 32) % (TK / 32) == 0, "one row per thread in TokStage");
  extern __shared__ __align__(128) float smem[];
  float* ring_mem = smem;
  float* s_ba = smem + 2 * WuSmem<TK>::STAGE;                 // bias partial sums of the row operand [TN]
  float* s_bb = s_ba + TN;                                    // ... of the column operand [TK]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_bb + TK);    // 2 mbarriers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  int pi = 0;
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (i < grp.nprob && (int)blockIdx.x >= grp.p[i].tile_begin) pi = i;
  const WuProblem& P = grp.p[pi];
  const int tile = blockIdx.x - P.tile_begin;
  const int r_base = (tile / P.tiles_c) * TN, c_base = (tile % P.tiles_c) * TK;
  const int rows_valid = min(TN, P.rows - r_base);
  const int m_begin = blockIdx.y * grp.MC;
  const int m_end = min(grp.M, m_begin + grp.MC);
  const int nchunk = (m_end - m_begin + KC - 1) / KC;
  const float* ga = P.a + r_base;
  const float* gb = P.b + c_base;
  const int lda = P.lda, ldb = P.ldb;
  const bool want_ba = P.bias_a != nullptr && c_base == 0;
  const bool want_bb = P.bias_b != nullptr && r_base == 0;

  if (tid == 0) {
    umma::mbar_init(bars, 1);
    umma::mbar_init(bars + 1, 1);
    umma::fence_mbar_init();
  }
  if (warp == 0) umma::tmem_alloc<TCOLS>(tmem_slot);
  for (int i = tid; i < TN + TK; i += RL_NT) s_ba[i] = 0.f;
  pdl_wait();      // the operands are written by the preceding kernels
  pdl_trigger();
  umma::tc_fence_before();
  __syncthreads();
  umma::tc_fence_after();
  const uint32_t tb = *tmem_slot;

  // register double buffer: the global loads of chunks j + 1 and j + 2 are in flight while chunk j is staged
  TokStage<TN> sa[2];
  TokStage<TK> sb[2];
  float bsum_a = 0.f, bsum_b = 0.f;
  Ring ring{bars, 0};
  constexpr uint32_t idesc = umma::idesc_tf32(TN, TK);
#pragma unroll
  for (int u = 0; u < 2; ++u)
    if (u < nchunk) {
      sa[u].load(ga, lda, rows_valid, m_begin + u * KC, m_end);
      sb[u].load(gb, ldb, TK, m_begin + u * KC, m_end);
    }
  auto step = [&](int j, TokStage<TN>& ra, TokStage<TK>& rb) {
    ring.wait_free();
    float* a_hi = ring_mem + ring.buf() * WuSmem<TK>::STAGE;
    float* a_lo = a_hi + TN * KC;
    float* b_hi = a_lo + TN * KC;
    float* b_lo = b_hi + TK * KC;
    ra.store(a_hi, a_lo);
    rb.store(b_hi, b_lo);
    if (want_ba) bsum_a += ra.token_sum();
    if (want_bb) bsum_b += rb.token_sum();
    if (j + 2 < nchunk) {
      ra.load(ga, lda, rows_valid, m_begin + (j + 2) * KC, m_end);
      rb.load(gb, ldb, TK, m_begin + (j + 2) * KC, m_end);
    }
    umma::fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      umma::tc_fence_after();
      umma::mma_chunk_3x<KC>(tb, a_hi, a_lo, KC, 0, b_hi, b_lo, idesc, j > 0 ? 1u : 0u);
      umma::commit(bars + ring.buf());
    }
    ++ring.chunk;
  };
  for (int j = 0; j < nchunk; j += 2) {
    step(j, sa[0], sb[0]);
    if (j + 1 < nchunk) step(j + 1, sa[1], sb[1]);
  }
  if constexpr (DET) {            // the warps holding the same rows add their sums in warp order
    for (int w = 0; w < RL_NT / 32; ++w) {
      if (warp == w) {
        if (want_ba && sa[0].active()) s_ba[sa[0].my_row()] += bsum_a;
        if (want_bb && sb[0].active()) s_bb[sb[0].my_row()] += bsum_b;
      }
      __syncthreads();
    }
  } else {
    if (want_ba && sa[0].active()) atomicAdd(&s_ba[sa[0].my_row()], bsum_a);
    if (want_bb && sb[0].active()) atomicAdd(&s_bb[sb[0].my_row()], bsum_b);
  }
  if (nchunk > 0) {
    ring.wait_last();
    umma::tc_fence_after();
    // epilogue: warp w reads TMEM lane quadrant w % 4 (tile rows 32 (w % 4) + lane); the 16-column groups of the tile
    // are dealt round-robin to the four warp groups w / 4
    const int quad = warp & 3, cgp = warp >> 2;
    const int row = quad * 32 + lane;
    // DET: out / bias_a / bias_b are partial slabs [token slice][rows x cols], slot = blockIdx.y
    float* orow = grad_slot<DET>(P.out, (size_t)P.rows * P.tiles_c * TK, blockIdx.y) + (size_t)(r_base + row) * P.so_r +
                  (size_t)c_base * P.so_c;
    const int so_c = P.so_c;
#pragma unroll
    for (int c16 = cgp; c16 < TK / 16; c16 += 4) {
      float t0[16];
      umma::tmem_ld16(umma::tmem_addr(tb, c16 * 16), t0);
      if (row < rows_valid) {
        if (so_c == 1) {
          // a thread owns 16 consecutive columns of its row: four 16-byte vector reductions (a quarter of the L2
          // transactions of scalar ones, which would touch 32 rows = 32 sectors per warp instruction)
#pragma unroll
          for (int i = 0; i < 16; i += 4) {
            if constexpr (DET)
              *reinterpret_cast<float4*>(orow + c16 * 16 + i) = make_float4(t0[i], t0[i + 1], t0[i + 2], t0[i + 3]);
            else
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(orow + c16 * 16 + i), "f"(t0[i]),
                           "f"(t0[i + 1]), "f"(t0[i + 2]), "f"(t0[i + 3])
                           : "memory");
          }
        } else {
          // transposed output: the lanes (rows of the tile) are contiguous in memory, one line per warp instruction
#pragma unroll
          for (int i = 0; i < 16; ++i) grad_add<DET>(orow + (size_t)(c16 * 16 + i) * so_c, t0[i]);
        }
      }
    }
  }
  umma::tc_fence_before();
  __syncthreads();
  if (want_ba && tid < rows_valid) grad_add<DET>(grad_slot<DET>(P.bias_a, P.rows, blockIdx.y) + r_base + tid, s_ba[tid]);
  if (want_bb && tid < TK) grad_add<DET>(grad_slot<DET>(P.bias_b, P.tiles_c * TK, blockIdx.y) + c_base + tid, s_bb[tid]);
  if (warp == 0) umma::tmem_dealloc<TCOLS>(tb);
}

template <int TK>
int launch(WuGroup& g, int total_tiles, cudaStream_t st, RlDet* det) {
  // one wave of CTAs (148 SMs), each with at least four chunks of tokens.  Measured on the training step (B = 256):
  // 112 / 148 / 222 / 296 CTAs -> 2.266 / 2.248 / 2.290 / 2.265 ms, 64 -> 2.355, 32 -> 2.425 (the in-order side stream
  // becomes the critical path); the SM time of these kernels (CTAs x duration) is the same at every split.
  int splits = (148 + total_tiles - 1) / total_tiles;
  const int max_splits = (g.M + 4 * KC - 1) / (4 * KC);
  if (splits > max_splits) splits = max_splits;
  if (det && splits > RL_DET_MAX_SPLIT) splits = RL_DET_MAX_SPLIT;
  if (splits < 1) splits = 1;
  int MC = (g.M + splits - 1) / splits;
  MC = ((MC + KC - 1) / KC) * KC;
  splits = (g.M + MC - 1) / MC;
  g.MC = MC;
  const size_t smem = WuSmem<TK>::BYTES;
  if (det == nullptr) {
    if (int rc = rl_set_smem(wgrad_umma_kernel<TK, false>, smem)) return rc;
    rl_launch_pdl(wgrad_umma_kernel<TK, false>, dim3(total_tiles, splits), dim3(RL_NT), smem, st, g);
    return rl_check_launch("wgrad_umma_kernel", TK, total_tiles);
  }
  for (int i = 0; i < g.nprob; ++i) {      // one partial slot per token slice
    WuProblem& p = g.p[i];
    const size_t cols = (size_t)p.tiles_c * TK;
    p.out = rl_det_take(det, p.out, (size_t)p.rows * cols, splits);
    p.bias_a = rl_det_take(det, p.bias_a, p.rows, splits);
    p.bias_b = rl_det_take(det, p.bias_b, cols, splits);
  }
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "wgrad: deterministic-mode workspace too small");
  for (int i = g.nprob; i < 4; ++i) g.p[i] = g.p[0];
  if (int rc = rl_set_smem(wgrad_umma_kernel<TK, true>, smem)) return rc;
  rl_launch_pdl(wgrad_umma_kernel<TK, true>, dim3(total_tiles, splits), dim3(RL_NT), smem, st, g);
  return rl_check_launch("wgrad_umma_kernel", TK, total_tiles);
}

int g_wgrad_umma = -1;
bool wgrad_umma_on() {
  if (g_wgrad_umma < 0) {
    const char* e = getenv("RALENET_WGRAD_UMMA");
    g_wgrad_umma = (e && *e) ? (atoi(e) != 0) : RL_WGRAD_UMMA_DEFAULT;
  }
  return g_wgrad_umma != 0;
}

}  // namespace

// 1: tcgen05 weight-gradient kernels (this file), 0: mma.sync kernels (wgrad.cu).  Same function; A/B switch.
extern "C" int ralenet_set_wgrad_umma(int on) {
  const int prev = wgrad_umma_on() ? 1 : 0;
  g_wgrad_umma = on ? 1 : 0;
  return prev;
}

// returns 1 if the group is not handled here (caller falls through to wgrad.cu)
int rl_launch_wgrad_group_umma(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det) {
  if (!wgrad_umma_on() || M < 4 * KC) return 1;
  WuGroup g;
  g.nprob = 0;
  g.M = M;
  int tiles = 0, TK = 0;
  for (int i = 0; i < n; ++i) {
    if (!d[i].dW) continue;
    if (g.nprob == 4) return 1;
    const int N = d[i].N, K = d[i].K;
    WuProblem& p = g.p[g.nprob];
    int rows, cols;
    if (N < TN && K >= TN) {                                   // few rows, many columns: tile the transpose
      p.a = d[i].X; p.lda = d[i].ldx; p.b = d[i].dY; p.ldb = d[i].ldy;
      p.out = d[i].dW; p.so_r = 1; p.so_c = K;
      p.bias_a = nullptr; p.bias_b = d[i].db;
      rows = K; cols = N;
    } else {
      p.a = d[i].dY; p.lda = d[i].ldy; p.b = d[i].X; p.ldb = d[i].ldx;
      p.out = d[i].dW; p.so_r = K; p.so_c = 1;
      p.bias_a = d[i].db; p.bias_b = nullptr;
      rows = N; cols = K;
    }
    const int tk = (cols % 128 == 0) ? 128 : cols;             // tile width of this problem
    if (tk != 32 && tk != 64 && tk != 128) return 1;
    if (TK == 0) TK = tk;
    if (tk != TK) return 1;                                    // one tile width per launch
    p.rows = rows;
    p.tiles_c = cols / tk;
    p.tile_begin = tiles;
    tiles += ((rows + TN - 1) / TN) * p.tiles_c;
    ++g.nprob;
  }
  if (g.nprob == 0) return RL_OK;
  for (int i = g.nprob; i < 4; ++i) g.p[i] = g.p[0];
  switch (TK) {
    case 32: return launch<32>(g, tiles, st, det);
    case 64: return launch<64>(g, tiles, st, det);
    case 128: return launch<128>(g, tiles, st, det);
  }
  return 1;
}
