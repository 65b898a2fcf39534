// umma.cuh -- tcgen05 (5th-generation tensor core) building blocks for the wide RA-LENet stages:
// TMEM allocation, un-swizzled K-major shared-memory matrix descriptors, kind::tf32 MMA issue with the
// 3-pass split (hi*hi + lo*hi + hi*lo, fp32-grade), mbarrier completion tracking and TMEM -> register loads.
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
// Staging of a ROWS x KC operand block whose contraction index is the ROW of the global matrix (dgrad: B = W^T) into a
// K-major tile pair (hi = x, lo = x - trunc(x)):   element (n, k) <- src[k * ld + n],  n < ROWS (multiple of 32),
// k < KC.  A warp reads 32 consecutive n of four consecutive k rows (4 x 128 contiguous bytes) and each lane writes one
// 16-byte chunk (its n, four k) of the K-major tile.  Split in two halves so that the global loads can be issued long
// before the tile buffer is free: load() pulls the block into registers, store() splits and writes it.  NT = threads of
// the CTA.
template <int ROWS, int KC, int NT>
struct TStage {
  static constexpr int NB = ROWS / 32, NQ = KC / 4, ITEMS = NB * NQ;
  static constexpr int PER = (ITEMS + NT / 32 - 1) / (NT / 32);
  static_assert(ROWS % 32 == 0 && KC % 4 == 0, "TStage: tile shape");
  float4 v[PER];

  __device__ __forceinline__ void load(const float* __restrict__ src, int ld) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int item = wid + i * (NT / 32);
      v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (item < ITEMS) {
        const int nb = item % NB, q = item / NB;
        const float* p = src + (size_t)(4 * q) * ld + nb * 32 + lane;
        v[i] = make_float4(__ldg(p), __ldg(p + ld), __ldg(p + 2 * (size_t)ld), __ldg(p + 3 * (size_t)ld));
      }
    }
  }
  __device__ __forceinline__ void store(float* hi, float* lo) const {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int item = wid + i * (NT / 32);
      if (item < ITEMS) {
        const int nb = item % NB, q = item / NB;
        const int n = nb * 32 + lane;
        const int o = (n & 7) * 4 + q * 32 + (n >> 3) * (NQ * 32);
        *reinterpret_cast<float4*>(hi + o) = v[i];
        *reinterpret_cast<float4*>(lo + o) = lo4(v[i]);
      }
    }
  }
};

}  // namespace umma
