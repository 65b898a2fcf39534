// wgrad.cu -- weight-gradient GEMM over the token dimension, split-K across CTAs.
//   dW[n*K + k] += sum_m dY[m*ldy + n] * X[m*ldx + k]        db[n] += sum_m dY[m*ldy + n]
// M = all tokens of the batch (B*L: 65536 ... 4096 at B=256), N,K in {4..512}.  The reduction dim is
// the long one, so each CTA owns a (TN x TK) output tile and a slice of MC tokens, accumulates in
// registers and finishes with fp32 red.global (atomicAdd).  HBM-bound: reads (N+K)*4 B per token.
#include "common.cuh"

namespace {

constexpr int MS = 32;   // tokens staged per inner step

template <int TN, int TK, bool DET>
__global__ void __launch_bounds__(RL_NT) wgrad_kernel(const float* __restrict__ dY, int ldy,
                                                      const float* __restrict__ X, int ldx, int M, int N, int K,
                                                      float* __restrict__ dW, float* __restrict__ db, int MC) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  constexpr int RM = (TN >= 16) ? TN / 16 : 1;
  constexpr int RN = (TK >= 16) ? TK / 16 : 1;
  constexpr int NTN = TK / RN;                 // threads along k
  constexpr int NTM = TN / RM;                 // threads along n
  constexpr int LDA = TN + 1, LDB = TK + 1;
  __shared__ float sA[MS * LDA];
  __shared__ float sB[MS * LDB];

  const int tiles_k = K / TK;
  const int tile_n = blockIdx.x / tiles_k, tile_k = blockIdx.x % tiles_k;
  const int n_base = tile_n * TN, k_base = tile_k * TK;
  const int m_begin = blockIdx.y * MC;
  const int m_end = min(M, m_begin + MC);

  const int tid = threadIdx.x;
  const bool active = tid < NTN * NTM;
  const int tn = tid % NTN, tm = tid / NTN;
  float acc[RM][RN];
#pragma unroll
  for (int i = 0; i < RM; ++i)
#pragma unroll
    for (int j = 0; j < RN; ++j) acc[i][j] = 0.f;
  float bacc = 0.f;
  const bool do_bias = (db != nullptr) && (tile_k == 0);

  for (int m0 = m_begin; m0 < m_end; m0 += MS) {
    const int rows = min(MS, m_end - m0);
    for (int i = tid; i < MS * TN; i += RL_NT) {
      const int c = i % TN, r = i / TN;
      sA[r * LDA + c] = (r < rows) ? __ldg(dY + (size_t)(m0 + r) * ldy + n_base + c) : 0.f;
    }
    for (int i = tid; i < MS * TK; i += RL_NT) {
      const int c = i % TK, r = i / TK;
      sB[r * LDB + c] = (r < rows) ? __ldg(X + (size_t)(m0 + r) * ldx + k_base + c) : 0.f;
    }
    __syncthreads();
    if (active) micro_gemm<RM, RN>(acc, sA, 1, LDA, sB, LDB, tm * RM, tn, NTN, MS);
    if (do_bias && tid < TN) {
#pragma unroll 8
      for (int r = 0; r < MS; ++r) bacc += sA[r * LDA + tid];
    }
    __syncthreads();
  }
  dW = grad_slot<DET>(dW, (size_t)N * K, blockIdx.y);       // DET: slot = token slice
  if (active) {
#pragma unroll
    for (int i = 0; i < RM; ++i)
#pragma unroll
      for (int j = 0; j < RN; ++j)
        grad_add<DET>(dW + (size_t)(n_base + tm * RM + i) * K + k_base + tn + j * NTN, acc[i][j]);
  }
  if (do_bias && tid < TN) grad_add<DET>(grad_slot<DET>(db, N, blockIdx.y) + n_base + tid, bacc);
}

template <int TN, int TK>
int launch(const float* dY, int ldy, const float* X, int ldx, int M, int N, int K, float* dW, float* db,
           cudaStream_t st, RlDet* det) {
  const int tiles = (N / TN) * (K / TK);
  // aim for ~4 CTAs per SM overall, but never slices shorter than 128 tokens
  int splits = (592 + tiles - 1) / tiles;
  const int max_splits = (M + 127) / 128;
  if (splits > max_splits) splits = max_splits;
  if (det && splits > RL_DET_MAX_SPLIT) splits = RL_DET_MAX_SPLIT;
  if (splits < 1) splits = 1;
  int MC = (M + splits - 1) / splits;
  MC = ((MC + MS - 1) / MS) * MS;
  splits = (M + MC - 1) / MC;
  dim3 grid(tiles, splits);
  if (det == nullptr) {
    rl_launch_pdl(wgrad_kernel<TN, TK, false>, dim3(grid), dim3(RL_NT), 0, st, dY, ldy, X, ldx, M, N, K, dW, db, MC);
    return rl_check_launch("wgrad_kernel", N, K);
  }
  dW = rl_det_take(det, dW, (size_t)N * K, splits);     // one partial slot per token slice
  db = rl_det_take(det, db, N, splits);
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "wgrad: deterministic-mode workspace too small");
  rl_launch_pdl(wgrad_kernel<TN, TK, true>, dim3(grid), dim3(RL_NT), 0, st, dY, ldy, X, ldx, M, N, K, dW, db, MC);
  return rl_check_launch("wgrad_kernel", N, K);
}

template <int TN>
int dispatch_k(int TK, const float* dY, int ldy, const float* X, int ldx, int M, int N, int K, float* dW, float* db,
               cudaStream_t st, RlDet* det) {
  switch (TK) {
    case 4: return launch<TN, 4>(dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 8: return launch<TN, 8>(dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 16: return launch<TN, 16>(dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 32: return launch<TN, 32>(dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 64: return launch<TN, 64>(dY, ldy, X, ldx, M, N, K, dW, db, st, det);
  }
  rl_set_error("wgrad: unsupported K tile %d", TK);
  return RL_ERR_SHAPE;
}

inline int pick_tile(int n) {
  if (n >= 64 && n % 64 == 0) return 64;
  if (n == 32 || n == 16 || n == 8 || n == 4) return n;
  return 0;
}

}  // namespace

// ---------------------------------------------------------------------------------------------
// Grouped tensor-core weight gradients: up to 4 (dY, X) -> dW problems that share the token dimension M
// (all weight matrices of one attention / feed-forward half) in ONE launch.  Each CTA owns a T x T tile of
// one dW and a slice of tokens; the token slice is streamed through a 2-stage cp.async pipeline and
// contracted with 3xTF32 mma.sync (A = dY^T in A_KM layout, B = X in B_KN layout); fp32 red.global at the end.
namespace {

struct WgProblem {
  const float* dY; const float* X; float* dW; float* db;
  int ldy, ldx, N, K, tile_begin, tiles_k;
};
struct WgGroup {
  WgProblem p[4];
  int nprob, M, MC;
};

constexpr int WG_MS = 64;   // tokens per pipeline stage

template <int T, bool DET>
__global__ void __launch_bounds__(RL_NT) wgrad_group_kernel(const WgGroup grp) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  constexpr int LD = T + 8;                     // % 32 in {8, 24}: conflict-free A_KM / B_KN fragment loads
  extern __shared__ __align__(16) float smem[];
  float* sA = smem;                             // [2][WG_MS][LD]  dY tile
  float* sB = smem + 2 * WG_MS * LD;            // [2][WG_MS][LD]  X tile
  const int tid = threadIdx.x;
  int pi = 0;
#pragma unroll
  for (int i = 1; i < 4; ++i)
    if (i < grp.nprob && (int)blockIdx.x >= grp.p[i].tile_begin) pi = i;
  const WgProblem& P = grp.p[pi];
  const int tile = blockIdx.x - P.tile_begin;
  const int n_base = (tile / P.tiles_k) * T, k_base = (tile % P.tiles_k) * T;
  const int m_begin = blockIdx.y * grp.MC;
  const int m_end = min(grp.M, m_begin + grp.MC);
  const int nst = (m_end - m_begin + WG_MS - 1) / WG_MS;
  const float* gA = P.dY + n_base;
  const float* gB = P.X + k_base;
  const int ldy = P.ldy, ldx = P.ldx;

  auto issue = [&](int st) {
    const int m0 = m_begin + st * WG_MS;
    float* dA = sA + (st & 1) * WG_MS * LD;
    float* dB = sB + (st & 1) * WG_MS * LD;
    constexpr int V = T / 4;                    // float4 per row
    for (int i = tid; i < WG_MS * V; i += RL_NT) {
      const int r = i / V, c = (i % V) * 4;
      const bool ok = (m0 + r) < m_end;
      const size_t row = ok ? (size_t)(m0 + r) : (size_t)m_begin;
      cp_async16_zfill(dA + r * LD + c, gA + row * ldy + c, ok);
      cp_async16_zfill(dB + r * LD + c, gB + row * ldx + c, ok);
    }
    cp_async_commit();
  };

  MmaTile<T, T> acc;
  acc.init();
  float bacc = 0.f;
  const bool do_bias = (P.db != nullptr) && (k_base == 0);
  if (nst > 0) issue(0);
  for (int st = 0; st < nst; ++st) {
    if (st + 1 < nst) {
      issue(st + 1);
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float* cA = sA + (st & 1) * WG_MS * LD;
    const float* cB = sB + (st & 1) * WG_MS * LD;
    acc.template mac<A_KM, B_KN>(cA, LD, cB, LD, WG_MS);
    if (do_bias && tid < T) {
#pragma unroll 8
      for (int r = 0; r < WG_MS; ++r) bacc += cA[r * LD + tid];
    }
    __syncthreads();
  }
  const int K = P.K;
  float* dW = grad_slot<DET>(P.dW, (size_t)P.N * K, blockIdx.y);     // DET: slot = token slice
  acc.epilogue([&](int n, int k, float v) { grad_add<DET>(dW + (size_t)(n_base + n) * K + k_base + k, v); });
  if (do_bias && tid < T) grad_add<DET>(grad_slot<DET>(P.db, P.N, blockIdx.y) + n_base + tid, bacc);
}

template <int T>
int launch_group(WgGroup& g, int total_tiles, cudaStream_t st, RlDet* det) {
  int splits = (444 + total_tiles - 1) / total_tiles;            // ~3 CTAs per SM overall
  const int max_splits = (g.M + 2 * WG_MS - 1) / (2 * WG_MS);    // at least 2 pipeline stages per CTA
  if (splits > max_splits) splits = max_splits;
  if (det && splits > RL_DET_MAX_SPLIT) splits = RL_DET_MAX_SPLIT;
  if (splits < 1) splits = 1;
  int MC = (g.M + splits - 1) / splits;
  MC = ((MC + WG_MS - 1) / WG_MS) * WG_MS;
  splits = (g.M + MC - 1) / MC;
  g.MC = MC;
  const size_t smem = sizeof(float) * 4 * WG_MS * (T + 8);
  dim3 grid(total_tiles, splits);
  if (det == nullptr) {
    if (int rc = rl_set_smem(wgrad_group_kernel<T, false>, smem)) return rc;
    rl_launch_pdl(wgrad_group_kernel<T, false>, dim3(grid), dim3(RL_NT), smem, st, g);
    return rl_check_launch("wgrad_group_kernel", T, total_tiles);
  }
  for (int i = 0; i < g.nprob; ++i) {      // one partial slot per token slice
    g.p[i].dW = rl_det_take(det, g.p[i].dW, (size_t)g.p[i].N * g.p[i].K, splits);
    g.p[i].db = rl_det_take(det, g.p[i].db, g.p[i].N, splits);
  }
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "wgrad: deterministic-mode workspace too small");
  for (int i = g.nprob; i < 4; ++i) g.p[i] = g.p[0];
  if (int rc = rl_set_smem(wgrad_group_kernel<T, true>, smem)) return rc;
  rl_launch_pdl(wgrad_group_kernel<T, true>, dim3(grid), dim3(RL_NT), smem, st, g);
  return rl_check_launch("wgrad_group_kernel", T, total_tiles);
}

}  // namespace

// up to 4 problems sharing M; dims must all be multiples of 32 for the tensor-core path, otherwise the
// problems are launched one by one on the FFMA kernel.
int rl_launch_wgrad_group_umma(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det);   // wgrad_umma.cu

int rl_launch_wgrad_group_reg(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det);    // wgrad_reg.cu

// det: deterministic mode, the GEMMs write partial slabs [token slice][N][K] recorded in *det
int rl_launch_wgrad_group(const RlWgradDesc* d, int n, int M, cudaStream_t st, RlDet* det) {
  {
    const int rc = rl_launch_wgrad_group_reg(d, n, M, st, det);     // register-tile kernel; 1: group not handled there
    if (rc <= 0) return rc;
  }
  {
    const int rc = rl_launch_wgrad_group_umma(d, n, M, st, det);    // tcgen05 kernels; 1: group not handled there
    if (rc <= 0) return rc;
  }
  int cnt = 0, mind = 1 << 30;
  bool aligned = true;
  for (int i = 0; i < n; ++i) {
    if (!d[i].dW) continue;
    ++cnt;
    mind = min(mind, min(d[i].N, d[i].K));
    aligned = aligned && (d[i].N % 32 == 0) && (d[i].K % 32 == 0) && (d[i].ldy % 4 == 0) && (d[i].ldx % 4 == 0) &&
              ((uintptr_t)d[i].dY % 16 == 0) && ((uintptr_t)d[i].X % 16 == 0);
  }
  if (cnt == 0) return RL_OK;
  if (!aligned || cnt > 4) {
    for (int i = 0; i < n; ++i)
      if (int rc = rl_launch_wgrad(d[i].dY, d[i].ldy, d[i].X, d[i].ldx, M, d[i].N, d[i].K, d[i].dW, d[i].db, st, det))
        return rc;
    return RL_OK;
  }
  const int T = (mind % 64 == 0) ? 64 : 32;
  WgGroup g;
  g.nprob = 0;
  g.M = M;
  int tiles = 0;
  for (int i = 0; i < n; ++i) {
    if (!d[i].dW) continue;
    WgProblem& p = g.p[g.nprob++];
    p.dY = d[i].dY; p.X = d[i].X; p.dW = d[i].dW; p.db = d[i].db;
    p.ldy = d[i].ldy; p.ldx = d[i].ldx; p.N = d[i].N; p.K = d[i].K;
    p.tile_begin = tiles;
    p.tiles_k = d[i].K / T;
    tiles += (d[i].N / T) * (d[i].K / T);
  }
  for (int i = g.nprob; i < 4; ++i) g.p[i] = g.p[0];
  return T == 64 ? launch_group<64>(g, tiles, st, det) : launch_group<32>(g, tiles, st, det);
}

int rl_launch_wgrad(const float* dY, int ldy, const float* X, int ldx, int M, int N, int K, float* dW, float* db,
                    cudaStream_t st, RlDet* det) {
  if (dW == nullptr) return RL_OK;
  const int TN = pick_tile(N), TK = pick_tile(K);
  RL_REQUIRE(TN && TK && M > 0, RL_ERR_SHAPE, "wgrad: unsupported shape M=%d N=%d K=%d", M, N, K);
  switch (TN) {
    case 4: return dispatch_k<4>(TK, dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 8: return dispatch_k<8>(TK, dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 16: return dispatch_k<16>(TK, dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 32: return dispatch_k<32>(TK, dY, ldy, X, ldx, M, N, K, dW, db, st, det);
    case 64: return dispatch_k<64>(TK, dY, ldy, X, ldx, M, N, K, dW, db, st, det);
  }
  return RL_ERR_SHAPE;
}

extern "C" int ralenet_wgrad(const float* dY, int32_t ldy, const float* X, int32_t ldx, int32_t M, int32_t N, int32_t K,
                             float* dW, float* db, void* stream) {
  RL_REQUIRE(dY && X && dW, RL_ERR_NULL, "wgrad: NULL tensor");
  return rl_launch_wgrad(dY, ldy, X, ldx, M, N, K, dW, db, (cudaStream_t)stream);
}
