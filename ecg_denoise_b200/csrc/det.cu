// det.cu -- deterministic mode (RL_NET_DETERMINISTIC): partial slabs and their batched reduction.
//
// Every cross-CTA accumulation into a parameter gradient of the whole-network backward becomes a plain store into
// its own slot of a partial slab [slots][n] (grad_add / grad_slot in common.cuh); the slot is a function of the work
// item alone (window, tile, token slice of a weight-gradient GEMM).  grad_reduce_kernel then sums the slots of every
// slab recorded for one backward kernel in slot order and adds the total to the gradient with one read-modify-write
// per element, so the result does not depend on how CTAs or streams are scheduled.
#include "common.cuh"

namespace {

struct RedGroup {
  RlGradRed r[RL_DET_MAXRED];
  int cta_begin[RL_DET_MAXRED + 1];
  int ew[RL_DET_MAXRED];      // elements per CTA (power of two <= 32); the RL_NT / ew thread groups split the slots
  int nred;
};

__global__ void __launch_bounds__(RL_NT) grad_reduce_kernel(const RedGroup g) {
  pdl_wait();
  pdl_trigger();
  __shared__ float s_part[RL_NT];
  int k = 0;
  while (k + 1 < g.nred && (int)blockIdx.x >= g.cta_begin[k + 1]) ++k;
  const RlGradRed& R = g.r[k];
  const int ew = g.ew[k], ng = RL_NT / ew;
  const int e = threadIdx.x % ew, grp = threadIdx.x / ew;
  const int i = ((int)blockIdx.x - g.cta_begin[k]) * ew + e;
  // group q sums the contiguous slot range [q * per, (q + 1) * per) in slot order; the ranges are added in group order
  const int per = (R.slots + ng - 1) / ng;
  const int s0 = grp * per, s1 = min(R.slots, s0 + per);
  float s = 0.f;
  if (i < R.n) {
    const float* p = R.src + (size_t)s0 * R.n + i;
#pragma unroll 8
    for (int q = s0; q < s1; ++q, p += R.n) s += __ldg(p);
  }
  s_part[threadIdx.x] = s;
  __syncthreads();
  if (grp == 0 && i < R.n) {
    float t = s_part[e];
    for (int q = 1; q < ng; ++q) t += s_part[q * ew + e];
    R.dst[i] += t;
  }
}

}  // namespace

float* rl_det_take(RlDet* d, float* g, size_t n, int slots) {
  if (g == nullptr || n == 0) return nullptr;
  const size_t need = ((n * (size_t)slots) + 3) & ~(size_t)3;
  if (d->nred >= RL_DET_MAXRED || d->used + need > d->cap || slots < 1) {
    rl_set_error("deterministic mode: partial slab overflow (%zu + %zu floats of %zu, %d slabs)", d->used, need, d->cap,
                 d->nred);
    d->nred = RL_DET_MAXRED + 1;      // poisoned: rl_det_ok() is false from now on
    return nullptr;
  }
  float* p = d->slab + d->used;
  d->used += need;
  d->red[d->nred++] = RlGradRed{p, g, (int)n, slots};
  return p;
}

bool rl_det_ok(const RlDet* d) { return d->nred <= RL_DET_MAXRED; }

int rl_launch_grad_reduce(RlDet* d, cudaStream_t st) {
  RL_REQUIRE(rl_det_ok(d), RL_ERR_SHAPE, "deterministic mode: partial slab overflow");
  if (d->nred == 0) return RL_OK;
  RedGroup g;
  g.nred = d->nred;
  int ctas = 0;
  for (int k = 0; k < d->nred; ++k) {
    g.r[k] = d->red[k];
    int ew = 1;
    while (ew < 32 && ew < d->red[k].n) ew *= 2;
    g.ew[k] = ew;
    g.cta_begin[k] = ctas;
    ctas += (d->red[k].n + ew - 1) / ew;
  }
  for (int k = d->nred; k <= RL_DET_MAXRED; ++k) g.cta_begin[k] = ctas;
  for (int k = d->nred; k < RL_DET_MAXRED; ++k) { g.r[k] = g.r[0]; g.ew[k] = g.ew[0]; }
  d->nred = 0;
  rl_launch_pdl(grad_reduce_kernel, dim3(ctas), dim3(RL_NT), 0, st, g);
  return rl_check_launch("grad_reduce_kernel", g.nred);
}
