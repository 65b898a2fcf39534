// tma.cuh -- Tensor Memory Accelerator staging of the weight operands of the tcgen05 kernels.
//
// A weight chunk (ROWS output rows x 32 contraction floats = ROWS x 128 bytes of a row-major [N][K] nn.Linear weight)
// is fetched by ONE elected thread with `cp.async.bulk.tensor.2d` (SASS: UTMALDG) into the canonical K-major
// SWIZZLE_128B shared-memory layout -- 8-row groups of 1024 bytes, the 16-byte chunks of row r XOR-swizzled by r % 8 --
// which the UMMA shared-memory descriptor names directly (layout type 2, SBO = 1024 B, K advance = 32 B per K = 8
// step inside the 128-byte atom).  Completion is tracked with an mbarrier transaction count.  The tf32 remainder
// tile (lo = x - trunc(x), the second operand of the 3-pass split) is derived from the landed tile element-wise, so
// the swizzle never has to be undone by a thread.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

// host (tma.cu): tensor map of a row-major fp32 matrix [rows][cols] (leading dimension ld floats), box = box_rows x 32
// floats, SWIZZLE_128B.  Cached per (pointer, shape); returns RL_OK or an RL_ERR_* code.
int rl_tmap_weight(const float* base, int rows, int cols, int ld, int box_rows, CUtensorMap* out);

namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// box at (c0 = first column, c1 = first row) -> dst; arrives on `bar` with the byte count
__device__ __forceinline__ void load_2d(void* dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
          smem_u32(dst)),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// UMMA shared-memory descriptor of a K-major SWIZZLE_128B tile (tile base 1024-byte aligned)
__device__ __forceinline__ uint64_t desc_sw128(uint32_t byte_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((byte_addr >> 4) & 0x3fff);
  d |= (uint64_t)1 << 16;                         // LBO: unused for swizzled K-major tiles
  d |= (uint64_t)(1024 >> 4) << 32;               // SBO: 8 rows x 128 bytes
  d |= (uint64_t)1 << 46;                         // descriptor version of sm_100
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
  return d;
}

}  // namespace tma

#include "umma.cuh"
namespace tma {
// D[tmem] (+)= A[:, k0:k0+KCW] * B^T with the 3-pass tf32 split; A: un-swizzled K-major tile pair (umma.cuh) with KT_A
// contraction elements per row, B: one KCW <= 32 wide chunk in the K-major SWIZZLE_128B layout written by TMA and its
// remainder tile in the same layout.  Issued by ONE thread.
// TF32 (inference precision RL_F_TF32): ONE pass, hi x hi, on operands rounded to tf32 (umma::rna4, derive_lo<NT, true>);
// the remainder tiles are neither written nor read.
template <int KCW, bool TF32 = false>
__device__ __forceinline__ void mma_chunk_3x(uint32_t tmem_d, const float* a_hi, const float* a_lo, int KT_A, int k0,
                                             const float* b_hi, const float* b_lo, uint32_t idesc, uint32_t accum) {
  static_assert(KCW % 8 == 0 && KCW <= 32, "one SWIZZLE_128B atom holds 32 contraction floats");
  const uint32_t sbo_a = (uint32_t)(KT_A / 4) * 128u;
  const uint32_t ah = umma::smem_u32(a_hi) + (uint32_t)(k0 / 4) * 128u, al = umma::smem_u32(a_lo) + (uint32_t)(k0 / 4) * 128u;
  const uint32_t bh = umma::smem_u32(b_hi), bl = umma::smem_u32(b_lo);
#pragma unroll
  for (int ks = 0; ks < KCW / 8; ++ks) {
    const uint64_t dah = umma::make_desc(ah + ks * 256u, 128u, sbo_a), dal = umma::make_desc(al + ks * 256u, 128u, sbo_a);
    const uint64_t dbh = desc_sw128(bh + ks * 32u), dbl = desc_sw128(bl + ks * 32u);
    if constexpr (TF32) {
      umma::mma_tf32(tmem_d, dah, dbh, idesc, accum);
    } else {
      umma::mma_tf32(tmem_d, dal, dbh, idesc, accum);
      umma::mma_tf32(tmem_d, dah, dbl, idesc, 1u);
      umma::mma_tf32(tmem_d, dah, dbh, idesc, 1u);
    }
    accum = 1u;
  }
}
// element-wise remainder tile of a landed chunk (any layout): lo = hi - trunc_tf32(hi); all NT threads of the CTA.
// TF32: the chunk is rounded to tf32 in place instead (same pass, same synchronisation point; lo is not touched).
template <int NT, bool TF32 = false>
__device__ __forceinline__ void derive_lo(float* hi, float* lo, int floats) {
  float4* h4 = reinterpret_cast<float4*>(hi);
  float4* l4 = reinterpret_cast<float4*>(lo);
  for (int i = threadIdx.x; i < floats / 4; i += NT) {
    const float4 v = h4[i];
    if constexpr (TF32) h4[i] = umma::rna4(v);
    else l4[i] = umma::lo4(v);
  }
}
}  // namespace tma
