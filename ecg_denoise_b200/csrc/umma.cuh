// umma.cuh -- tcgen05 (5th-generation tensor core) building blocks for the wide RA-LENet stages:
// TMEM allocation, un-swizzled K-major shared-memory matrix descriptors, kind::tf32 MMA issue with the
// 3-pass split (hi*hi + lo*hi + hi*lo, fp32-grade), mbarrier completion tracking and TMEM -> register loads; and
// the phases the tile kernels share: operand staging into the K-major layout, TMEM -> shared partial tiles and their
// reduction across a cluster.
//
// Facts verified on B200 with tools/umma_probe.cu (gpurun_out/umma_probe1.txt, summarised in profiles/):
//   * kind::tf32 reads the fp32 container and ignores the low 13 mantissa bits (matches a truncating
//     reference to 1e-6), so x and lo = x - trunc(x) can be fed as they are;
//   * canonical un-swizzled K-major tile: core matrix = 8 rows x 16 bytes stored contiguously (128 B);
//     descriptor LBO = byte stride between the two 16-byte K chunks of one K = 8 MMA, SBO = byte stride
//     between 8-row groups;
//   * accumulator of an M = 128 MMA: row i -> TMEM lane i; M = 64: row i -> lane (i / 16) * 32 + i % 16;
//     column j -> column j (fp32).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <cooperative_groups.h>
#include "common.cuh"

namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t make_desc(uint32_t byte_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((byte_addr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;
  d |= (uint64_t)1 << 46;     // descriptor version of sm_100
  return d;                   // layout_type 0 (no swizzle), base_offset 0
}

// instruction descriptor: D fp32, A/B tf32, both K-major, M x N tile
__host__ __device__ constexpr uint32_t idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(da), "l"(db), "r"(idesc), "r"(accum)
      : "memory");
}

// D[tmem] (+)= A[:, k0:k0+KC] * B[:, 0:KC]^T with the 3-pass split.  a_hi/a_lo: K-major tile with KT_A elements
// per row (the chunk starts at element k0); b_hi/b_lo: K-major tile holding exactly the KC-wide chunk.
// Issued by ONE thread.  `accum` = 0 overwrites the accumulator with the first MMA.
template <int KC>
__device__ __forceinline__ void mma_chunk_3x(uint32_t tmem_d, const float* a_hi, const float* a_lo, int KT_A, int k0,
                                             const float* b_hi, const float* b_lo, uint32_t idesc, uint32_t accum) {
  const uint32_t sbo_a = (uint32_t)(KT_A / 4) * 128u, sbo_b = (uint32_t)(KC / 4) * 128u;
  const uint32_t ah = smem_u32(a_hi) + (uint32_t)(k0 / 4) * 128u, al = smem_u32(a_lo) + (uint32_t)(k0 / 4) * 128u;
  const uint32_t bh = smem_u32(b_hi), bl = smem_u32(b_lo);
#pragma unroll
  for (int ks = 0; ks < KC / 8; ++ks) {
    const uint64_t dah = make_desc(ah + ks * 256u, 128u, sbo_a), dal = make_desc(al + ks * 256u, 128u, sbo_a);
    const uint64_t dbh = make_desc(bh + ks * 256u, 128u, sbo_b), dbl = make_desc(bl + ks * 256u, 128u, sbo_b);
    mma_tf32(tmem_d, dal, dbh, idesc, accum);
    mma_tf32(tmem_d, dah, dbl, idesc, 1u);
    mma_tf32(tmem_d, dah, dbh, idesc, 1u);
    accum = 1u;
  }
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// arrives on `bar` once every tcgen05 operation issued so far by this thread has completed
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// wait for the phase of `bar` with the given parity; traps instead of hanging if it never completes
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t done = 0;
  for (uint32_t it = 0; !done; ++it) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(done)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    if (it > (1u << 26)) __trap();
  }
}

// issue-side bookkeeping of the 2-deep weight ring: buffer b = chunk & 1 may be overwritten once the MMAs of the
// chunk that used it two steps ago have completed (one commit per chunk on bar[b])
struct Ring {
  uint64_t* bar;
  int chunk;
  __device__ __forceinline__ int buf() const { return chunk & 1; }
  __device__ __forceinline__ void wait_free() const {
    if (chunk >= 2) mbar_wait(bar + (chunk & 1), (uint32_t)(((chunk >> 1) - 1) & 1));
  }
  // wait until the MMAs of the most recently issued chunk (and everything before it) are complete
  __device__ __forceinline__ void wait_last() const {
    const int last = chunk - 1;
    mbar_wait(bar + (last & 1), (uint32_t)((last >> 1) & 1));
  }
};

__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// one full warp allocates NCOLS (power of two >= 32) TMEM columns; the base address lands in *slot (shared)
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(NCOLS) : "memory");
}

// TMEM -> registers: the calling warp reads its lane quadrant (warp % 4), one row per thread, N consecutive columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  __syncwarp();
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// address of (lane quadrant of the calling warp, column col) relative to the allocation base
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, int col) {
  const uint32_t quad = (threadIdx.x >> 5) & 3u;
  return base + ((quad * 32u) << 16) + (uint32_t)col;
}

__device__ __forceinline__ float trunc_tf32(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }
// single-pass operand (RL_F_TF32): four values rounded to nearest (ties away) to tf32, stored in the fp32 container
__device__ __forceinline__ float4 rna4(float4 v) {
  uint32_t r0, r1, r2, r3;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r0) : "f"(v.x));
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r1) : "f"(v.y));
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r2) : "f"(v.z));
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r3) : "f"(v.w));
  return make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float(r2), __uint_as_float(r3));
}
// tf32 remainder of four values, v - trunc_tf32(v), with two packed subtractions (Blackwell `sub.f32x2`, SASS FADD2)
__device__ __forceinline__ float4 lo4(float4 v) {
  const float t0 = trunc_tf32(v.x), t1 = trunc_tf32(v.y), t2 = trunc_tf32(v.z), t3 = trunc_tf32(v.w);
  float4 r;
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tsub.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r.x), "=f"(r.y)
      : "f"(v.x), "f"(v.y), "f"(t0), "f"(t1));
  asm("{\n\t.reg .b64 a, b, c;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tsub.f32x2 c, a, b;\n\t"
      "mov.b64 {%0, %1}, c;\n\t}"
      : "=f"(r.z), "=f"(r.w)
      : "f"(v.z), "f"(v.w), "f"(t2), "f"(t3));
  return r;
}


// ---------------------------------------------------------------------------------------------
// The un-swizzled K-major core-matrix layout of the staged tiles (the `make_desc` strides of mma_chunk_3x: LBO = 128 B,
// SBO = KT / 4 * 128 B): offset in floats of the 16-byte chunk (row 8 g + r, elements [4 q, 4 q + 4)) of a tile with
// KT contraction elements per row.
__device__ __forceinline__ int kmajor_off(int g, int r, int q, int KT) { return r * 4 + q * 32 + g * (KT / 4) * 32; }

// four values of a tile pair at offset o: hi = v, lo = its tf32 remainder; TF32 (single pass): hi = v rounded to tf32
template <bool TF32 = false>
__device__ __forceinline__ void store_pair(float* hi, float* lo, int o, float4 v) {
  if constexpr (TF32) {
    *reinterpret_cast<float4*>(hi + o) = rna4(v);
  } else {
    *reinterpret_cast<float4*>(hi + o) = v;
    *reinterpret_cast<float4*>(lo + o) = lo4(v);
  }
}

// Rows -> A tile: the TM = 128 rows of src (row-major, KT floats per row; rows >= nvalid staged as zeros) into a
// K-major tile pair with KT elements per row, by the 16 warps of the CTA.  A warp owns 8 rows; lane = (row % 8,
// 16-byte chunk % 4), so global reads cover full sectors and the tile stores are contiguous.  `norm`: each 16-byte
// chunk v of row `row` first becomes pre(v, row, chunk), then the row is layer-normalised with the affine
// s_ln = weight [KT] | bias [KT] staged in shared memory.
template <int KT, bool TF32, typename Pre>
__device__ __forceinline__ void stage_rows(float* hi, float* lo, const float* __restrict__ src, int nvalid, bool norm,
                                           const float* s_ln, Pre pre) {
  constexpr int NI = KT / 16;                                // chunks per lane
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int rsub = lane & 7, qsub = lane >> 3;
  const int row = warp * 8 + rsub;
  const bool ok = row < nvalid;
  float4 v[NI];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int qc = qsub + 4 * i;
    v[i] = ok ? __ldg(reinterpret_cast<const float4*>(src + (size_t)row * KT) + qc) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (norm) v[i] = pre(v[i], row, qc);
    s += v[i].x + v[i].y + v[i].z + v[i].w;
  }
  float mu = 0.f, rstd = 1.f;
  if (norm) {
    s += __shfl_xor_sync(0xffffffffu, s, 8);
    s += __shfl_xor_sync(0xffffffffu, s, 16);
    mu = s * (1.0f / KT);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NI; ++i) {
      const float d0 = v[i].x - mu, d1 = v[i].y - mu, d2 = v[i].z - mu, d3 = v[i].w - mu;
      q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
    }
    q += __shfl_xor_sync(0xffffffffu, q, 8);
    q += __shfl_xor_sync(0xffffffffu, q, 16);
    rstd = rsqrtf(q * (1.0f / KT) + RL_LN_EPS);
  }
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int qc = qsub + 4 * i;
    float4 u = v[i];
    if (norm) {
      const float4 w4 = *reinterpret_cast<const float4*>(s_ln + 4 * qc);
      const float4 b4 = *reinterpret_cast<const float4*>(s_ln + KT + 4 * qc);
      u.x = fmaf((v[i].x - mu) * rstd, w4.x, b4.x);
      u.y = fmaf((v[i].y - mu) * rstd, w4.y, b4.y);
      u.z = fmaf((v[i].z - mu) * rstd, w4.z, b4.z);
      u.w = fmaf((v[i].w - mu) * rstd, w4.w, b4.w);
      if (!ok) u = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    store_pair<TF32>(hi, lo, kmajor_off(warp, rsub, qc, KT), u);
  }
}

// Accumulator -> shared memory: the TM = 128 x C fp32 tile at TMEM column col into sp [TM][C + 4].  Warp w reads its
// lane quadrant w % 4 (row 32 (w % 4) + lane = threadIdx.x % 128) and the C / 4 columns of group w / 4.
template <int C>
__device__ __forceinline__ void tmem_to_smem(float* sp, uint32_t tmem_base, int col) {
  constexpr int LDP = C + 4, CW = C / 4;                     // row stride, columns per warp group (16 or 32)
  const int row = threadIdx.x & 127, cgp = threadIdx.x >> 7;
#pragma unroll
  for (int c16 = 0; c16 < CW; c16 += 16) {
    float t0[16];
    tmem_ld16(tmem_addr(tmem_base, col + cgp * CW + c16), t0);
#pragma unroll
    for (int i = 0; i < 16; i += 4)
      *reinterpret_cast<float4*>(sp + row * LDP + cgp * CW + c16 + i) = make_float4(t0[i], t0[i + 1], t0[i + 2], t0[i + 3]);
  }
}

// sum of the NSL partial tiles of a cluster (part[q] = tile of CTA rank q, 16-byte DSMEM loads) at offset off
template <int NSL>
__device__ __forceinline__ float4 dsmem_sum4(const float* const (&part)[NSL], int off) {
  float4 s = *reinterpret_cast<const float4*>(part[0] + off);
#pragma unroll
  for (int q = 1; q < NSL; ++q) {
    const float4 p = *reinterpret_cast<const float4*>(part[q] + off);
    s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
  }
  return s;
}

// Reduction of the partial output tiles [TM][C + 4] of a cluster of NSL CTAs, y = sum of the partials + bias
// (+ residual) (+ extra): CTA r finishes rows [r RPC, (r + 1) RPC).  load() fetches the bias and residual terms of
// those rows before the cluster barrier instead of one round trip per item behind it; store() sums and writes them.
template <int TM, int C, int NSL>
struct ClusterReduce {
  static constexpr int RPC = TM / NSL, RIT = RPC * (C / 4) / RL_NT;  // rows finished per CTA, float4 items per thread
  static_assert(RPC * (C / 4) % RL_NT == 0, "reduce: items must tile the CTA");
  float4 add4[RIT];

  // bias [C] or NULL; x (added if resid), extra (or NULL): [tokens][C]; rows of the tile start at token tok0
  __device__ __forceinline__ void load(int r, int nvalid, size_t tok0, const float* bias, const float* x, bool resid,
                                       const float* extra) {
#pragma unroll
    for (int it = 0; it < RIT; ++it) {
      const int i = threadIdx.x + it * RL_NT;
      const int rr = r * RPC + i / (C / 4), c = (i % (C / 4)) * 4;
      add4[it] = bias ? __ldg(reinterpret_cast<const float4*>(bias + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
      if (rr < nvalid) {
        const size_t g = (tok0 + rr) * C + c;
        if (resid) {
          const float4 x4 = __ldg(reinterpret_cast<const float4*>(x + g));
          add4[it].x += x4.x; add4[it].y += x4.y; add4[it].z += x4.z; add4[it].w += x4.w;
        }
        if (extra) {
          const float4 e4 = __ldg(reinterpret_cast<const float4*>(extra + g));
          add4[it].x += e4.x; add4[it].y += e4.y; add4[it].z += e4.z; add4[it].w += e4.w;
        }
      }
    }
  }
  // after the cluster barrier: sp = this CTA's partial tile (the same offset in every CTA of the cluster)
  __device__ __forceinline__ void store(cooperative_groups::cluster_group& cluster, float* sp, int r, int nvalid,
                                        size_t tok0, float* y) const {
    const float* part[NSL];
#pragma unroll
    for (int q = 0; q < NSL; ++q) part[q] = cluster.map_shared_rank(sp, q);
#pragma unroll
    for (int it = 0; it < RIT; ++it) {
      const int i = threadIdx.x + it * RL_NT;
      const int rr = r * RPC + i / (C / 4), c = (i % (C / 4)) * 4;
      if (rr >= nvalid) continue;
      float4 s = dsmem_sum4<NSL>(part, rr * (C + 4) + c);
      s.x += add4[it].x; s.y += add4[it].y; s.z += add4[it].z; s.w += add4[it].w;
      *reinterpret_cast<float4*>(y + (tok0 + rr) * C + c) = s;
    }
  }
};

// ---------------------------------------------------------------------------------------------
// Staging of a ROWS x KC operand block whose contraction index is the ROW of the global matrix (dgrad: B = W^T; the
// weight gradients: both operands, contraction over the tokens) into a K-major tile pair (hi = x, lo = x - trunc(x)):
// element (n, k) <- src[k * ld + n],  n < ROWS (multiple of 32), k < KC.  A warp reads 32 consecutive n of four
// consecutive k rows (4 x 128 contiguous bytes) and each lane writes one 16-byte chunk (its n, four k) of the K-major
// tile.  Split in two halves so that the global loads can be issued long before the tile buffer is free: load() pulls
// the block into registers, store() splits and writes it.  NT = threads of the CTA.  GUARD: rows n >= rows_valid and
// k >= m_end - m0 are staged as zeros.
template <int ROWS, int KC, int NT, bool GUARD = false>
struct TStage {
  static constexpr int NB = ROWS / 32, NQ = KC / 4, ITEMS = NB * NQ;
  static constexpr int PER = (ITEMS + NT / 32 - 1) / (NT / 32);
  static_assert(ROWS % 32 == 0 && KC % 4 == 0, "TStage: tile shape");
  float4 v[PER];

  // src -> element (n = 0, k = m0)
  __device__ __forceinline__ void load(const float* __restrict__ src, int ld, int rows_valid = ROWS, int m0 = 0,
                                       int m_end = KC) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int item = wid + i * (NT / 32);
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (item < ITEMS) {
        const int nb = item % NB, q = item / NB;
        const int n = nb * 32 + lane, m = m0 + 4 * q;
        if (!GUARD || n < rows_valid) {
          const float* p = src + (size_t)m * ld + n;
          if (!GUARD || m + 3 < m_end) {
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
      const int item = wid + i * (NT / 32);
      if (item < ITEMS) {
        const int n = (item % NB) * 32 + lane;
        store_pair(hi, lo, kmajor_off(n >> 3, n & 7, item / NB, KC), v[i]);
      }
    }
  }
  // sum over the staged k of the row this thread holds (every item of a thread has the same row: (NT / 32) % NB == 0)
  __device__ __forceinline__ float token_sum() const {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    return s;
  }
  __device__ __forceinline__ int my_row() const { return ((threadIdx.x >> 5) % NB) * 32 + (threadIdx.x & 31); }
  __device__ __forceinline__ bool active() const { return (int)(threadIdx.x >> 5) < ITEMS; }
};

}  // namespace umma
