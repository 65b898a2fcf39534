// stem_head.cu -- the Conv1d/BatchNorm stem, the Conv1d head, the MSE loss + SNR/RMSE metrics, the
// k=13 lead-mixing convolutions of the 12-lead wrapper, and flat Adam.  All HBM-bound, one CTA per window.
//
// Reference: model/transformer.py:570-574, 623 (stem), :617-619, 664-667 (head);
// denoise_train.py:53 (mse_loss), :24,57 (Adam); local_utils/evaluate.py:27-29, 49-51 (RMSE, SNR);
// model/ralenet_12leads.py:684-709 (newrale convs).
#include "common.cuh"

namespace {

constexpr int MAXL = 512;

// conv(2->8,k3,p1) + LeakyReLU(0.2) at position t from a zero-haloed smem copy of the 2 x L input
__device__ __forceinline__ void stem_conv(const float* sx /*[2][L+2]*/, int L, int t, const float* w /*[48]*/,
                                          const float* b, float* c /*[8] pre-activation*/) {
  const float x00 = sx[t], x01 = sx[t + 1], x02 = sx[t + 2];
  const float x10 = sx[L + 2 + t], x11 = sx[L + 2 + t + 1], x12 = sx[L + 2 + t + 2];
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float* wo = w + o * 6;
    c[o] = b[o] + wo[0] * x00 + wo[1] * x01 + wo[2] * x02 + wo[3] * x10 + wo[4] * x11 + wo[5] * x12;
  }
}
__device__ __forceinline__ float lrelu(float v, float s) { return v > 0.f ? v : v * s; }

__device__ __forceinline__ void load_stem_window(float* sx, float* sw, float* sb, const float* x, const float* w,
                                                 const float* b, int L) {
  const int tid = threadIdx.x;
  for (int i = tid; i < 2 * (L + 2); i += RL_NT) {
    const int ch = i / (L + 2), p = i % (L + 2) - 1;
    sx[i] = (p >= 0 && p < L) ? __ldg(x + ch * L + p) : 0.f;
  }
  if (tid < 48) sw[tid] = __ldg(w + tid);
  if (tid < 8) sb[tid] = __ldg(b + tid);
}

// per-window partial sums of a and a^2 per channel -> partials[b][16]
__global__ void __launch_bounds__(RL_NT) stem_stats_kernel(const rl_stem_args a) {
  __shared__ float sx[2 * (MAXL + 2)];
  __shared__ float sw[48], sb[8];
  const int L = a.L, tid = threadIdx.x;
  load_stem_window(sx, sw, sb, a.x + (size_t)blockIdx.x * 2 * L, a.conv_w, a.conv_b, L);
  __syncthreads();
  float s1[8], s2[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) s1[o] = s2[o] = 0.f;
  for (int t = tid; t < L; t += RL_NT) {
    float c[8];
    stem_conv(sx, L, t, sw, sb, c);
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      const float v = lrelu(c[o], 0.2f);
      s1[o] += v;
      s2[o] += v * v;
    }
  }
  // warp sums meet in shared memory and are added in warp order: the BatchNorm statistics -- and with them the
  // training-mode forward -- are bit-reproducible from run to run (shared-memory atomics were not)
  __shared__ float swp[RL_NT / 32][16];
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float r1 = warp_sum(s1[o]), r2 = warp_sum(s2[o]);
    if ((tid & 31) == 0) {
      swp[tid >> 5][o] = r1;
      swp[tid >> 5][8 + o] = r2;
    }
  }
  __syncthreads();
  if (tid < 16) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < RL_NT / 32; ++w) tot += swp[w][tid];
    a.partials[(size_t)blockIdx.x * 16 + tid] = tot;
  }
}

// sum partials[B][16] in double -> out[16] (+ optional extras); one CTA
__global__ void __launch_bounds__(RL_NT) reduce16_kernel(const float* __restrict__ partials, int B, float* out,
                                                         float count_or_neg, float* add_a, float* add_b) {
  __shared__ double sd[RL_NT];
  const int tid = threadIdx.x, j = tid % 16, r = tid / 16;
  double s = 0.0;
  for (int b = r; b < B; b += RL_NT / 16) s += (double)partials[(size_t)b * 16 + j];
  sd[tid] = s;
  __syncthreads();
  if (tid < 16) {
    double tot = 0.0;
    for (int k = 0; k < RL_NT / 16; ++k) tot += sd[k * 16 + tid];
    out[tid] = (float)tot;
    if (add_a && tid >= 8) atomicAdd(add_a + tid - 8, (float)tot);   // d_bn_w += sum g*ahat
    if (add_b && tid < 8) atomicAdd(add_b + tid, (float)tot);        // d_bn_b += sum g
  }
  if (tid == 0 && count_or_neg >= 0.f) out[16] = count_or_neg;
}

__global__ void __launch_bounds__(RL_NT) stem_apply_kernel(const rl_stem_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float sx[2 * (MAXL + 2)];
  __shared__ float sw[48], sb[8], smu[8], srs[8], sgam[8], sbet[8];
  const int L = a.L, tid = threadIdx.x;
  load_stem_window(sx, sw, sb, a.x + (size_t)blockIdx.x * 2 * L, a.conv_w, a.conv_b, L);
  if (tid < 8) {
    float mu, var;
    if (a.training) {
      const float n = a.stats[16];
      mu = a.stats[tid] / n;
      var = fmaxf(a.stats[8 + tid] / n - mu * mu, 0.f);
      if (blockIdx.x == 0) {             // running statistics (momentum 0.1, unbiased variance)
        a.running_mean[tid] = (1.f - a.momentum) * a.running_mean[tid] + a.momentum * mu;
        a.running_var[tid] = (1.f - a.momentum) * a.running_var[tid] + a.momentum * var * (n / (n - 1.f));
        if (tid == 0 && a.num_batches_tracked) *a.num_batches_tracked += 1;
      }
    } else {
      mu = a.running_mean[tid];
      var = a.running_var[tid];
    }
    smu[tid] = mu;
    srs[tid] = rsqrtf(var + a.eps);
    sgam[tid] = __ldg(a.bn_w + tid);
    sbet[tid] = __ldg(a.bn_b + tid);
  }
  __syncthreads();
  float* yw = a.y + (size_t)blockIdx.x * L * 8;
  for (int t = tid; t < L; t += RL_NT) {
    float c[8];
    stem_conv(sx, L, t, sw, sb, c);
#pragma unroll
    for (int o = 0; o < 8; ++o) c[o] = (lrelu(c[o], 0.2f) - smu[o]) * srs[o] * sgam[o] + sbet[o];
    float4* y4 = reinterpret_cast<float4*>(yw + t * 8);
    y4[0] = make_float4(c[0], c[1], c[2], c[3]);
    y4[1] = make_float4(c[4], c[5], c[6], c[7]);
  }
}

__device__ __forceinline__ void stem_mu_rstd(const rl_stem_bwd_args& a, int o, float& mu, float& rstd) {
  if (a.training) {
    const float n = a.stats[16];
    mu = a.stats[o] / n;
    rstd = rsqrtf(fmaxf(a.stats[8 + o] / n - mu * mu, 0.f) + a.eps);
  } else {
    mu = 0.f;   // not needed: ahat only enters the training-mode terms and d_bn_w (handled by caller)
    rstd = rsqrtf(a.running_var[o] + a.eps);
  }
}

// per-window sums of g and g*ahat per channel -> partials[b][16]  ([0:8] = sum g, [8:16] = sum g*ahat)
__global__ void __launch_bounds__(RL_NT) stem_bwd_stats_kernel(const rl_stem_bwd_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float sx[2 * (MAXL + 2)];
  __shared__ float sw[48], sb[8], smu[8], srs[8];
  const int L = a.L, tid = threadIdx.x;
  load_stem_window(sx, sw, sb, a.x + (size_t)blockIdx.x * 2 * L, a.conv_w, a.conv_b, L);
  if (tid < 8) {
    float mu, rs;
    stem_mu_rstd(a, tid, mu, rs);
    if (!a.training) mu = a.running_mean[tid];
    smu[tid] = mu;
    srs[tid] = rs;
  }
  __syncthreads();
  const float* gw = a.g + (size_t)blockIdx.x * L * 8;
  const float* g2w = a.g2 ? a.g2 + (size_t)blockIdx.x * L * 8 : nullptr;
  float s1[8], s2[8];
#pragma unroll
  for (int o = 0; o < 8; ++o) s1[o] = s2[o] = 0.f;
  for (int t = tid; t < L; t += RL_NT) {
    float c[8];
    stem_conv(sx, L, t, sw, sb, c);
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      float g = __ldg(gw + t * 8 + o);
      if (g2w) g += __ldg(g2w + t * 8 + o);
      const float ah = (lrelu(c[o], 0.2f) - smu[o]) * srs[o];
      s1[o] += g;
      s2[o] += g * ah;
    }
  }
  // warp sums meet in shared memory and are added in warp order: the BatchNorm statistics -- and with them the
  // training-mode forward -- are bit-reproducible from run to run (shared-memory atomics were not)
  __shared__ float swp[RL_NT / 32][16];
#pragma unroll
  for (int o = 0; o < 8; ++o) {
    const float r1 = warp_sum(s1[o]), r2 = warp_sum(s2[o]);
    if ((tid & 31) == 0) {
      swp[tid >> 5][o] = r1;
      swp[tid >> 5][8 + o] = r2;
    }
  }
  __syncthreads();
  if (tid < 16) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < RL_NT / 32; ++w) tot += swp[w][tid];
    a.partials[(size_t)blockIdx.x * 16 + tid] = tot;
  }
}

template <bool DET>
__global__ void __launch_bounds__(RL_NT) stem_bwd_apply_kernel(const rl_stem_bwd_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float sx[2 * (MAXL + 2)];
  __shared__ float sdc[8 * (MAXL + 2)];
  __shared__ float sw[48], sb[8], smu[8], srs[8], sgam[8], sm1[8], sm2[8];
  const int L = a.L, tid = threadIdx.x;
  load_stem_window(sx, sw, sb, a.x + (size_t)blockIdx.x * 2 * L, a.conv_w, a.conv_b, L);
  if (tid < 8) {
    float mu, rs;
    stem_mu_rstd(a, tid, mu, rs);
    if (!a.training) mu = a.running_mean[tid];
    smu[tid] = mu;
    srs[tid] = rs;
    const float gam = __ldg(a.bn_w + tid);
    sgam[tid] = gam;
    if (a.training) {
      const float n = a.stats[16];
      sm1[tid] = gam * a.sums[tid] / n;          // mean(dahat)
      sm2[tid] = gam * a.sums[8 + tid] / n;      // mean(dahat * ahat)
    } else {
      sm1[tid] = 0.f;
      sm2[tid] = 0.f;
    }
  }
  for (int i = tid; i < 8 * (L + 2); i += RL_NT) sdc[i] = 0.f;
  __syncthreads();
  const float* gw = a.g + (size_t)blockIdx.x * L * 8;
  const float* g2w = a.g2 ? a.g2 + (size_t)blockIdx.x * L * 8 : nullptr;
  const bool train = a.training;
  for (int t = tid; t < L; t += RL_NT) {
    float c[8];
    stem_conv(sx, L, t, sw, sb, c);
#pragma unroll
    for (int o = 0; o < 8; ++o) {
      float g = __ldg(gw + t * 8 + o);
      if (g2w) g += __ldg(g2w + t * 8 + o);
      const float ah = (lrelu(c[o], 0.2f) - smu[o]) * srs[o];
      const float dah = g * sgam[o];
      const float da = train ? srs[o] * (dah - sm1[o] - ah * sm2[o]) : dah * srs[o];
      const float dc = da * (c[o] > 0.f ? 1.f : 0.2f);
      sdc[o * (L + 2) + t + 1] = dc;
    }
  }
  __syncthreads();
  if (a.d_conv_w) {
    // dW[o][i][k] = sum_t dc[o][t] x[i][t+k-1], db[o] = sum_t dc[o][t], from the two shared-memory tiles: thread =
    // (one of the 56 sums, one of 8 token segments), the 8 segments of a sum sit in neighbouring lanes (3 shuffles),
    // one red.global per sum and CTA.  (Round 2 kept 56 partial sums per token thread and pushed each through a
    // 5-step warp reduction plus a shared-memory atomic: 60 % of the samples of head_bwd, ncu r2_v38.)
    const int seg = tid & 7;                               // tokens seg, seg + 8, ...: neighbouring lanes, neighbouring words
    for (int jb = 0; jb < 56; jb += RL_NT >> 3) {          // (same trip count for every thread: full-warp shuffles)
      const int j = jb + (tid >> 3);
      float acc = 0.f;
      if (j < 48) {
        const int o = j / 6, i = (j % 6) / 3, k = j % 3;
        const float* pd = sdc + o * (L + 2) + 1;
        const float* px = sx + i * (L + 2) + k;
        for (int t = seg; t < L; t += 8) acc = fmaf(pd[t], px[t], acc);
      } else if (j < 56) {
        const float* pd = sdc + (j - 48) * (L + 2) + 1;
        for (int t = seg; t < L; t += 8) acc += pd[t];
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (seg == 0 && j < 56)        // DET: d_conv_w / d_conv_b are partial slabs [B][48] / [B][8]
        grad_add<DET>(j < 48 ? grad_slot<DET>(a.d_conv_w, 48, blockIdx.x) + j
                             : grad_slot<DET>(a.d_conv_b, 8, blockIdx.x) + j - 48, acc);
    }
  }
  if (a.dx) {   // dx[i][t] = sum_{o,k} dc[o][t-k+1] w[o][i][k]
    float* dxw = a.dx + (size_t)blockIdx.x * 2 * L;
    for (int idx = tid; idx < 2 * L; idx += RL_NT) {
      const int i = idx / L, t = idx % L;
      float s = 0.f;
#pragma unroll
      for (int o = 0; o < 8; ++o)
#pragma unroll
        for (int k = 0; k < 3; ++k) s = fmaf(sdc[o * (L + 2) + (t - k + 1) + 1], sw[o * 6 + i * 3 + k], s);
      dxw[idx] = s;
    }
  }
}

// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(RL_NT) head_fwd_kernel(const rl_head_fwd_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float ss[(MAXL + 2) * 8];
  __shared__ float sw[48], sb[2];
  const int L = a.L, tid = threadIdx.x;
  const float* xw = a.x + (size_t)blockIdx.x * L * 8;
  const float* kw = a.skip ? a.skip + (size_t)blockIdx.x * L * 8 : nullptr;
  for (int i = tid; i < (L + 2) * 8; i += RL_NT) {
    const int t = i / 8 - 1;
    float v = 0.f;
    if (t >= 0 && t < L) {
      v = __ldg(xw + t * 8 + (i % 8));
      if (kw) v += __ldg(kw + t * 8 + (i % 8));
    }
    ss[i] = v;
  }
  if (tid < 48) sw[tid] = __ldg(a.w + tid);
  if (tid < 2) sb[tid] = __ldg(a.b + tid);
  __syncthreads();
  float* ow = a.out + (size_t)blockIdx.x * 2 * L;
  for (int idx = tid; idx < 2 * L; idx += RL_NT) {
    const int o = idx / L, t = idx % L;
    float s = sb[o];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int k = 0; k < 3; ++k) s = fmaf(sw[o * 24 + i * 3 + k], ss[(t + k) * 8 + i], s);
    ow[idx] = s;
  }
}

template <bool DET>
__global__ void __launch_bounds__(RL_NT) head_bwd_kernel(const rl_head_bwd_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float ss[(MAXL + 2) * 8];
  __shared__ float sdo[2 * (MAXL + 2)];
  __shared__ float sw[48];
  const int L = a.L, tid = threadIdx.x;
  const float* xw = a.x + (size_t)blockIdx.x * L * 8;
  const float* kw = a.skip ? a.skip + (size_t)blockIdx.x * L * 8 : nullptr;
  const float* dw = a.dout + (size_t)blockIdx.x * 2 * L;
  for (int i = tid; i < (L + 2) * 8; i += RL_NT) {
    const int t = i / 8 - 1;
    float v = 0.f;
    if (t >= 0 && t < L) {
      v = __ldg(xw + t * 8 + (i % 8));
      if (kw) v += __ldg(kw + t * 8 + (i % 8));
    }
    ss[i] = v;
  }
  for (int i = tid; i < 2 * (L + 2); i += RL_NT) {
    const int o = i / (L + 2), p = i % (L + 2) - 1;
    sdo[i] = (p >= 0 && p < L) ? __ldg(dw + o * L + p) : 0.f;
  }
  if (tid < 48) sw[tid] = __ldg(a.w + tid);
  __syncthreads();
  // ds[t][i] = sum_{o,k} dout[o][t-k+1] w[o][i][k]
  float* dsw = a.ds + (size_t)blockIdx.x * L * 8;
  for (int idx = tid; idx < L * 8; idx += RL_NT) {
    const int t = idx / 8, i = idx % 8;
    float s = 0.f;
#pragma unroll
    for (int o = 0; o < 2; ++o)
#pragma unroll
      for (int k = 0; k < 3; ++k) s = fmaf(sdo[o * (L + 2) + (t - k + 1) + 1], sw[o * 24 + i * 3 + k], s);
    dsw[idx] = s;
  }
  if (a.d_w) {
    // dW[o][i][k] = sum_t dout[o][t] s[t+k-1][i], db[o] = sum_t dout[o][t]: thread = (one of the 50 sums, one of 8
    // token segments); 3 shuffles join the segments, one red.global per sum and CTA (see stem_bwd_apply_kernel)
    const int seg = tid & 7;                               // tokens seg, seg + 8, ...
    for (int jb = 0; jb < 50; jb += RL_NT >> 3) {          // (same trip count for every thread: full-warp shuffles)
      const int j = jb + (tid >> 3);
      float acc = 0.f;
      if (j < 48) {
        const int o = j / 24, i = (j % 24) / 3, k = j % 3;
        const float* pd = sdo + o * (L + 2) + 1;
        const float* ps = ss + k * 8 + i;
        for (int t = seg; t < L; t += 8) acc = fmaf(pd[t], ps[t * 8], acc);
      } else if (j < 50) {
        const float* pd = sdo + (j - 48) * (L + 2) + 1;
        for (int t = seg; t < L; t += 8) acc += pd[t];
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if (seg == 0 && j < 50)        // DET: d_w / d_b are partial slabs [B][48] / [B][2]
        grad_add<DET>(j < 48 ? grad_slot<DET>(a.d_w, 48, blockIdx.x) + j : grad_slot<DET>(a.d_b, 2, blockIdx.x) + j - 48,
                      acc);
    }
  }
}

// ---------------------------------------------------------------------------------------------
template <bool DET>
__global__ void __launch_bounds__(RL_NT) mse_kernel(const rl_mse_args a) {
  pdl_wait();      // programmatic dependent launch: the previous kernel on the stream has completed
  pdl_trigger();   // let the next kernel get scheduled while this one runs
  __shared__ float s_red[32];
  const int per = a.per, tid = threadIdx.x;
  const size_t off = (size_t)blockIdx.x * per;
  float se = 0.f, sw = 0.f, st = 0.f;
  const float k = 2.f * a.inv_count * a.gscale;
  for (int i = tid; i < per; i += RL_NT) {
    const float t = __ldg(a.target + off + i);
    const float d = __ldg(a.pred + off + i) - t;
    const float w = a.weight ? __ldg(a.weight + i) : 1.f;
    se += d * d;
    sw += w * d * d;
    st += t * t;
    if (a.dout) a.dout[off + i] = k * w * d;
  }
  se = block_sum(se, s_red);
  sw = block_sum(sw, s_red);
  st = block_sum(st, s_red);
  if (tid == 0) {
    if (DET) a.partials[blockIdx.x] = sw * a.inv_count;      // summed in window order by grad_reduce_kernel
    else atomicAdd(a.loss, sw * a.inv_count);
    if (a.rmse) a.rmse[blockIdx.x] = sqrtf(se / per);
    if (a.snr) a.snr[blockIdx.x] = 10.f * log10f(st / se);
  }
}

// block-wide fp64 sum in a fixed shuffle / warp order (all RL_NT threads must call); result valid in every thread
__device__ __forceinline__ double block_sum_f64(double v, double* s_red /* >= 32 doubles */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) s_red[w] = v;
  __syncthreads();
  double r = (lane < (RL_NT >> 5)) ? s_red[lane] : 0.0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  return r;
}

// one CTA per window: (1, snr_in, snr_out, rmse) of local_utils/evaluate.py in fp64 -> partials[b][4]
__global__ void __launch_bounds__(RL_NT) eval_window_kernel(const rl_eval_args a) {
  pdl_wait();
  pdl_trigger();
  __shared__ double s_red[32];
  const int b = blockIdx.x, tid = threadIdx.x, per = a.per;
  double* out = a.partials + 4 * (size_t)b;
  if (__ldg(a.level + b) < 0) {            // tail slot of the evaluation draw: no window
    if (tid < 4) out[tid] = 0.0;
    if (tid == 0) {
      if (a.snr_in) a.snr_in[b] = 0.f;
      if (a.snr_out) a.snr_out[b] = 0.f;
      if (a.rmse) a.rmse[b] = 0.f;
    }
    return;
  }
  const size_t off = (size_t)b * per;
  double sy = 0.0, se = 0.0, sn = 0.0;
  for (int i = tid; i < per; i += RL_NT) {
    const double y = __ldg(a.clean + off + i);
    const double e = y - (double)__ldg(a.pred + off + i), n = y - (double)__ldg(a.noisy + off + i);
    sy = fma(y, y, sy);
    se = fma(e, e, se);
    sn = fma(n, n, sn);
  }
  sy = block_sum_f64(sy, s_red);
  se = block_sum_f64(se, s_red);
  sn = block_sum_f64(sn, s_red);
  if (tid == 0) {
    const double snr_in = 10.0 * log10(sy / sn), snr_out = 10.0 * log10(sy / se), rmse = sqrt(se / per);
    out[0] = 1.0;
    out[1] = snr_in;
    out[2] = snr_out;
    out[3] = rmse;
    if (a.snr_in) a.snr_in[b] = (float)snr_in;
    if (a.snr_out) a.snr_out[b] = (float)snr_out;
    if (a.rmse) a.rmse[b] = (float)rmse;
  }
}

// one CTA: acc[l][k] += sum over the windows b of level l of partials[b][k], in a fixed order (thread t takes
// b = t, t + RL_NT, ... in turn, then block_sum_f64); then the batch counter moves on
__global__ void __launch_bounds__(RL_NT) eval_reduce_kernel(const rl_eval_args a) {
  pdl_wait();
  pdl_trigger();
  __shared__ double s_red[32];
  for (int l = 0; l < a.n_snr; ++l) {
    double s[4] = {0.0, 0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < a.B; b += RL_NT) {
      if (__ldg(a.level + b) != l) continue;
      const double* p = a.partials + 4 * (size_t)b;
#pragma unroll
      for (int k = 0; k < 4; ++k) s[k] += p[k];
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const double v = block_sum_f64(s[k], s_red);
      if (threadIdx.x == 0) a.acc[4 * l + k] += v;
    }
  }
  if (threadIdx.x == 0 && a.counter) *a.counter += 1;
}

// ---------------------------------------------------------------------------------------------
// generic small Conv1d ('same', odd K) for the 12-lead wrapper; one CTA per window.
constexpr int CONV_MAX_CI = 12, CONV_MAX_K = 13;

__global__ void __launch_bounds__(RL_NT) conv1d_fwd_kernel(const rl_conv_fwd_args a) {
  extern __shared__ __align__(16) float smem[];
  const int L = a.L, Ci = a.Cin, Co = a.Cout, K = a.K, pad = a.K / 2, LP = L + 2 * pad;
  float* sx = smem;                      // [Ci][LP]
  float* sw = sx + Ci * LP;              // [Co][Ci][K]
  const int tid = threadIdx.x;
  const float* xw = a.x + (size_t)blockIdx.x * Ci * L;
  for (int i = tid; i < Ci * LP; i += RL_NT) {
    const int ch = i / LP, p = i % LP - pad;
    sx[i] = (p >= 0 && p < L) ? __ldg(xw + ch * L + p) : 0.f;
  }
  for (int i = tid; i < Co * Ci * K; i += RL_NT) sw[i] = __ldg(a.w + i);
  __syncthreads();
  float* yw = a.y + (size_t)blockIdx.x * Co * L;
  for (int idx = tid; idx < Co * L; idx += RL_NT) {
    const int o = idx / L, t = idx % L;
    float s = a.b ? __ldg(a.b + o) : 0.f;
    for (int i = 0; i < Ci; ++i) {
      const float* xr = sx + i * LP + t;
      const float* wr = sw + (o * Ci + i) * K;
      for (int k = 0; k < K; ++k) s = fmaf(wr[k], xr[k], s);
    }
    yw[idx] = a.act ? lrelu(s, a.slope) : s;
  }
}

// DET: d_w / d_b are partial slabs [B][Cout*Cin*K] / [B][Cout] (grad_add); one thread sums each element of a
// window's dW and db, so the slot of a CTA is its window
template <bool DET>
__global__ void __launch_bounds__(RL_NT) conv1d_bwd_kernel(const rl_conv_bwd_args a) {
  extern __shared__ __align__(16) float smem[];
  const int L = a.L, Ci = a.Cin, Co = a.Cout, K = a.K, pad = a.K / 2, LP = L + 2 * pad;
  float* sx = smem;                      // [Ci][LP]
  float* sdc = sx + Ci * LP;             // [Co][LP]  gradient w.r.t. pre-activation, zero halo
  float* sw = sdc + Co * LP;             // [Co][Ci][K]
  const int tid = threadIdx.x;
  const float* xw = a.x + (size_t)blockIdx.x * Ci * L;
  const float* dyw = a.dy + (size_t)blockIdx.x * Co * L;
  for (int i = tid; i < Ci * LP; i += RL_NT) {
    const int ch = i / LP, p = i % LP - pad;
    sx[i] = (p >= 0 && p < L) ? __ldg(xw + ch * L + p) : 0.f;
  }
  for (int i = tid; i < Co * Ci * K; i += RL_NT) sw[i] = __ldg(a.w + i);
  for (int i = tid; i < Co * LP; i += RL_NT) sdc[i] = 0.f;
  __syncthreads();
  for (int idx = tid; idx < Co * L; idx += RL_NT) {
    const int o = idx / L, t = idx % L;
    float d = __ldg(dyw + idx);
    if (a.act) {   // recompute the pre-activation sign
      float s = a.b ? __ldg(a.b + o) : 0.f;
      for (int i = 0; i < Ci; ++i) {
        const float* xr = sx + i * LP + t;
        const float* wr = sw + (o * Ci + i) * K;
        for (int k = 0; k < K; ++k) s = fmaf(wr[k], xr[k], s);
      }
      if (!(s > 0.f)) d *= a.slope;
    }
    sdc[o * LP + t + pad] = d;
  }
  __syncthreads();
  if (a.dx) {   // dx[i][t] = sum_{o,k} dc[o][t-k+pad] w[o][i][k]
    float* dxw = a.dx + (size_t)blockIdx.x * Ci * L;
    for (int idx = tid; idx < Ci * L; idx += RL_NT) {
      const int i = idx / L, t = idx % L;
      float s = 0.f;
      for (int o = 0; o < Co; ++o) {
        const float* dr = sdc + o * LP + t + 2 * pad;     // index (t - k + pad) + pad
        const float* wr = sw + (o * Ci + i) * K;
        for (int k = 0; k < K; ++k) s = fmaf(dr[-k], wr[k], s);
      }
      dxw[idx] = s;
    }
  }
  if (a.d_w) {  // dW[o][i][k] += sum_t dc[o][t] x[i][t+k-pad]
    float* const d_w = grad_slot<DET>(a.d_w, (size_t)Co * Ci * K, blockIdx.x);
    for (int idx = tid; idx < Co * Ci * K; idx += RL_NT) {
      const int k = idx % K, i = (idx / K) % Ci, o = idx / (K * Ci);
      const float* dr = sdc + o * LP + pad;
      const float* xr = sx + i * LP + k;
      float s = 0.f;
      for (int t = 0; t < L; ++t) s = fmaf(dr[t], xr[t], s);
      grad_add<DET>(d_w + idx, s);
    }
    if (a.d_b) {
      float* const d_b = grad_slot<DET>(a.d_b, Co, blockIdx.x);
      for (int o = tid; o < Co; o += RL_NT) {
        float s = 0.f;
        for (int t = 0; t < L; ++t) s += sdc[o * LP + pad + t];
        grad_add<DET>(d_b + o, s);
      }
    }
  }
}

__global__ void __launch_bounds__(RL_NT) adam_kernel(float* __restrict__ p, const float* __restrict__ g,
                                                     float* __restrict__ m, float* __restrict__ v, int64_t n, float lr,
                                                     float b1, float b2, float eps, float bc1, float bc2_sqrt,
                                                     float gscale, const int32_t* __restrict__ step_dev) {
  if (step_dev) {   // graph-replayable variant: bias corrections from the device-side step counter
    const float s = (float)(*step_dev);
    bc1 = 1.f - powf(b1, s);
    bc2_sqrt = sqrtf(1.f - powf(b2, s));
  }
  const int64_t i0 = ((int64_t)blockIdx.x * RL_NT + threadIdx.x) * 4;
  if (i0 + 3 < n) {
    float4 p4 = *reinterpret_cast<float4*>(p + i0);
    const float4 g4 = *reinterpret_cast<const float4*>(g + i0);
    float4 m4 = *reinterpret_cast<float4*>(m + i0);
    float4 v4 = *reinterpret_cast<float4*>(v + i0);
    float* pp = &p4.x;
    const float* gg = &g4.x;
    float* mm = &m4.x;
    float* vv = &v4.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gr = gg[k] * gscale;
      mm[k] = b1 * mm[k] + (1.f - b1) * gr;
      vv[k] = b2 * vv[k] + (1.f - b2) * gr * gr;
      pp[k] -= (lr / bc1) * mm[k] / (sqrtf(vv[k]) / bc2_sqrt + eps);
    }
    *reinterpret_cast<float4*>(p + i0) = p4;
    *reinterpret_cast<float4*>(m + i0) = m4;
    *reinterpret_cast<float4*>(v + i0) = v4;
  } else {
    for (int64_t i = i0; i < n; ++i) {
      const float gr = g[i] * gscale;
      m[i] = b1 * m[i] + (1.f - b1) * gr;
      v[i] = b2 * v[i] + (1.f - b2) * gr * gr;
      p[i] -= (lr / bc1) * m[i] / (sqrtf(v[i]) / bc2_sqrt + eps);
    }
  }
}

int check_BL(const char* who, int B, int L) {
  RL_REQUIRE(B > 0 && L > 0 && L <= MAXL, RL_ERR_SHAPE, "%s: unsupported B=%d L=%d (L <= %d)", who, B, L, MAXL);
  return RL_OK;
}

}  // namespace

extern "C" int ralenet_stem_stats(const rl_stem_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "stem_stats: args is NULL");
  if (int rc = check_BL("stem_stats", a->B, a->L)) return rc;
  RL_REQUIRE(a->x && a->conv_w && a->conv_b && a->stats && a->partials, RL_ERR_NULL, "stem_stats: NULL tensor");
  cudaStream_t st = (cudaStream_t)stream;
  rl_prof_pre(st);
  stem_stats_kernel<<<a->B, RL_NT, 0, st>>>(*a);
  if (int rc = rl_check_launch("stem_stats_kernel")) return rc;
  rl_prof_pre(st);
  reduce16_kernel<<<1, RL_NT, 0, st>>>(a->partials, a->B, a->stats, (float)a->B * (float)a->L, nullptr, nullptr);
  return rl_check_launch("reduce16_kernel");
}

extern "C" int ralenet_stem_apply(const rl_stem_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "stem_apply: args is NULL");
  if (int rc = check_BL("stem_apply", a->B, a->L)) return rc;
  RL_REQUIRE(a->x && a->conv_w && a->conv_b && a->bn_w && a->bn_b && a->y && a->running_mean && a->running_var,
             RL_ERR_NULL, "stem_apply: NULL tensor");
  RL_REQUIRE(!a->training || a->stats, RL_ERR_NULL, "stem_apply: training needs stats");
  rl_launch_pdl(stem_apply_kernel, dim3(a->B), dim3(RL_NT), 0, (cudaStream_t)stream, *a);
  return rl_check_launch("stem_apply_kernel");
}

extern "C" int ralenet_stem_bwd_stats(const rl_stem_bwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "stem_bwd_stats: args is NULL");
  if (int rc = check_BL("stem_bwd_stats", a->B, a->L)) return rc;
  RL_REQUIRE(a->g && a->x && a->conv_w && a->conv_b && a->sums && a->partials, RL_ERR_NULL,
             "stem_bwd_stats: NULL tensor");
  RL_REQUIRE(a->training ? (a->stats != nullptr) : (a->running_var && a->running_mean), RL_ERR_NULL,
             "stem_bwd_stats: needs stats (training) or running stats (eval)");
  cudaStream_t st = (cudaStream_t)stream;
  rl_launch_pdl(stem_bwd_stats_kernel, dim3(a->B), dim3(RL_NT), 0, st, *a);
  if (int rc = rl_check_launch("stem_bwd_stats_kernel")) return rc;
  rl_prof_pre(st);
  reduce16_kernel<<<1, RL_NT, 0, st>>>(a->partials, a->B, a->sums, -1.f, a->d_bn_w, a->d_bn_b);
  return rl_check_launch("reduce16_kernel");
}

int rl_stem_bwd_apply(const rl_stem_bwd_args* a, cudaStream_t st, RlDet* det) {
  RL_REQUIRE(a, RL_ERR_NULL, "stem_bwd_apply: args is NULL");
  if (int rc = check_BL("stem_bwd_apply", a->B, a->L)) return rc;
  RL_REQUIRE(a->g && a->x && a->conv_w && a->conv_b && a->bn_w && a->sums, RL_ERR_NULL, "stem_bwd_apply: NULL tensor");
  RL_REQUIRE(a->training ? (a->stats != nullptr) : (a->running_var && a->running_mean), RL_ERR_NULL,
             "stem_bwd_apply: needs stats (training) or running stats (eval)");
  RL_REQUIRE(!a->d_conv_w == !a->d_conv_b, RL_ERR_NULL, "stem_bwd_apply: d_conv_w/d_conv_b both or neither");
  if (det == nullptr) {
    rl_launch_pdl(stem_bwd_apply_kernel<false>, dim3(a->B), dim3(RL_NT), 0, st, *a);
    return rl_check_launch("stem_bwd_apply_kernel");
  }
  rl_stem_bwd_args d = *a;                     // one partial slot per window (CTA)
  d.d_conv_w = rl_det_take(det, a->d_conv_w, 48, a->B);
  d.d_conv_b = rl_det_take(det, a->d_conv_b, 8, a->B);
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "stem_bwd_apply: deterministic-mode workspace too small");
  rl_launch_pdl(stem_bwd_apply_kernel<true>, dim3(a->B), dim3(RL_NT), 0, st, d);
  if (int rc = rl_check_launch("stem_bwd_apply_kernel")) return rc;
  return rl_launch_grad_reduce(det, st);
}

extern "C" int ralenet_stem_bwd_apply(const rl_stem_bwd_args* a, void* stream) {
  return rl_stem_bwd_apply(a, (cudaStream_t)stream);
}

extern "C" int ralenet_head_fwd(const rl_head_fwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "head_fwd: args is NULL");
  if (int rc = check_BL("head_fwd", a->B, a->L)) return rc;
  RL_REQUIRE(a->x && a->w && a->b && a->out, RL_ERR_NULL, "head_fwd: NULL tensor");
  rl_launch_pdl(head_fwd_kernel, dim3(a->B), dim3(RL_NT), 0, (cudaStream_t)stream, *a);
  return rl_check_launch("head_fwd_kernel");
}

int rl_head_bwd(const rl_head_bwd_args* a, cudaStream_t st, RlDet* det) {
  RL_REQUIRE(a, RL_ERR_NULL, "head_bwd: args is NULL");
  if (int rc = check_BL("head_bwd", a->B, a->L)) return rc;
  RL_REQUIRE(a->dout && a->x && a->w && a->ds, RL_ERR_NULL, "head_bwd: NULL tensor");
  RL_REQUIRE(!a->d_w == !a->d_b, RL_ERR_NULL, "head_bwd: d_w/d_b both or neither");
  if (det == nullptr) {
    rl_launch_pdl(head_bwd_kernel<false>, dim3(a->B), dim3(RL_NT), 0, st, *a);
    return rl_check_launch("head_bwd_kernel");
  }
  rl_head_bwd_args d = *a;                     // one partial slot per window (CTA)
  d.d_w = rl_det_take(det, a->d_w, 48, a->B);
  d.d_b = rl_det_take(det, a->d_b, 2, a->B);
  RL_REQUIRE(rl_det_ok(det), RL_ERR_SHAPE, "head_bwd: deterministic-mode workspace too small");
  rl_launch_pdl(head_bwd_kernel<true>, dim3(a->B), dim3(RL_NT), 0, st, d);
  if (int rc = rl_check_launch("head_bwd_kernel")) return rc;
  return rl_launch_grad_reduce(det, st);
}

extern "C" int ralenet_head_bwd(const rl_head_bwd_args* a, void* stream) { return rl_head_bwd(a, (cudaStream_t)stream); }

extern "C" int ralenet_mse(const rl_mse_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "mse: args is NULL");
  RL_REQUIRE(a->B > 0 && a->per > 0, RL_ERR_SHAPE, "mse: B=%d per=%d", a->B, a->per);
  RL_REQUIRE(a->pred && a->target && a->loss, RL_ERR_NULL, "mse: NULL tensor");
  const cudaStream_t st = (cudaStream_t)stream;
  if (a->partials == nullptr) {
    rl_launch_pdl(mse_kernel<false>, dim3(a->B), dim3(RL_NT), 0, st, *a);
    return rl_check_launch("mse_kernel");
  }
  rl_launch_pdl(mse_kernel<true>, dim3(a->B), dim3(RL_NT), 0, st, *a);
  if (int rc = rl_check_launch("mse_kernel")) return rc;
  RlDet det = {a->partials, (size_t)((a->B + 3) & ~3), 0, {}, 0};     // the per-window sums, added in window order
  rl_det_take(&det, a->loss, 1, a->B);
  return rl_launch_grad_reduce(&det, st);
}

extern "C" int ralenet_eval_metrics(const rl_eval_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "eval_metrics: args is NULL");
  RL_REQUIRE(a->B > 0 && a->per > 0 && a->n_snr >= 1, RL_ERR_SHAPE, "eval_metrics: B=%d per=%d n_snr=%d", a->B, a->per,
             a->n_snr);
  RL_REQUIRE(a->clean && a->noisy && a->pred && a->level && a->partials && a->acc, RL_ERR_NULL,
             "eval_metrics: NULL tensor");
  const cudaStream_t st = (cudaStream_t)stream;
  rl_launch_pdl(eval_window_kernel, dim3(a->B), dim3(RL_NT), 0, st, *a);
  if (int rc = rl_check_launch("eval_window_kernel")) return rc;
  rl_launch_pdl(eval_reduce_kernel, dim3(1), dim3(RL_NT), 0, st, *a);
  return rl_check_launch("eval_reduce_kernel");
}

// tensor-core implicit-GEMM path for the k = 13 layers of newrale (conv_mma.cu)
bool rl_conv13_eligible(int L, int Ci, int Co, int K);
int rl_conv13_fwd_mma(const rl_conv_fwd_args* a, cudaStream_t st);
int rl_conv13_bwd_mma(const rl_conv_bwd_args* a, cudaStream_t st, bool det);

static int conv_check(int B, int L, int Ci, int Co, int K, size_t* smem, bool bwd) {
  RL_REQUIRE(B > 0 && L > 0 && L <= 8192 && Ci > 0 && Co > 0 && Ci <= CONV_MAX_CI && Co <= CONV_MAX_CI && K % 2 == 1 &&
                 K <= CONV_MAX_K,
             RL_ERR_SHAPE, "conv1d: unsupported B=%d L=%d Cin=%d Cout=%d K=%d", B, L, Ci, Co, K);
  const size_t LP = L + K - 1;
  *smem = sizeof(float) * (Ci * LP + (bwd ? Co * LP : 0) + (size_t)Co * Ci * K);
  RL_REQUIRE(*smem <= 200 * 1024, RL_ERR_SHAPE, "conv1d: window too long for shared memory (L=%d)", L);
  return RL_OK;
}

extern "C" int ralenet_conv1d_fwd(const rl_conv_fwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "conv1d_fwd: args is NULL");
  size_t smem = 0;
  if (int rc = conv_check(a->B, a->L, a->Cin, a->Cout, a->K, &smem, false)) return rc;
  RL_REQUIRE(a->x && a->w && a->y, RL_ERR_NULL, "conv1d_fwd: NULL tensor");
  if (rl_conv13_eligible(a->L, a->Cin, a->Cout, a->K)) return rl_conv13_fwd_mma(a, (cudaStream_t)stream);
  if (int rc = rl_set_smem(conv1d_fwd_kernel, smem)) return rc;
  rl_prof_pre((cudaStream_t)stream);
  conv1d_fwd_kernel<<<a->B, RL_NT, smem, (cudaStream_t)stream>>>(*a);
  return rl_check_launch("conv1d_fwd_kernel");
}

template <bool DET>
static int conv1d_bwd_launch(const rl_conv_bwd_args* a, size_t smem, cudaStream_t st) {
  if (rl_conv13_eligible(a->L, a->Cin, a->Cout, a->K)) return rl_conv13_bwd_mma(a, st, DET);
  if (int rc = rl_set_smem(conv1d_bwd_kernel<DET>, smem)) return rc;
  rl_prof_pre(st);
  conv1d_bwd_kernel<DET><<<a->B, RL_NT, smem, st>>>(*a);
  return rl_check_launch("conv1d_bwd_kernel");
}

extern "C" int ralenet_conv1d_bwd(const rl_conv_bwd_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "conv1d_bwd: args is NULL");
  size_t smem = 0;
  if (int rc = conv_check(a->B, a->L, a->Cin, a->Cout, a->K, &smem, true)) return rc;
  RL_REQUIRE(a->dy && a->x && a->w, RL_ERR_NULL, "conv1d_bwd: NULL tensor");
  return conv1d_bwd_launch<false>(a, smem, (cudaStream_t)stream);
}

extern "C" uint64_t ralenet_conv1d_slab_bytes(int32_t B, int32_t Cin, int32_t Cout, int32_t K) {
  if (B <= 0 || Cin <= 0 || Cout <= 0 || K <= 0) return 0;
  const uint64_t nw = (uint64_t)B * Cout * Cin * K, nb = (uint64_t)B * Cout;   // rl_det_take's 16-byte rounding
  return sizeof(float) * (((nw + 3) & ~(uint64_t)3) + ((nb + 3) & ~(uint64_t)3));
}

extern "C" int ralenet_conv1d_bwd_det(const rl_conv_bwd_args* a, float* slab, uint64_t slab_bytes, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "conv1d_bwd_det: args is NULL");
  size_t smem = 0;
  if (int rc = conv_check(a->B, a->L, a->Cin, a->Cout, a->K, &smem, true)) return rc;
  RL_REQUIRE(a->dy && a->x && a->w && slab, RL_ERR_NULL, "conv1d_bwd_det: NULL tensor or slab");
  const uint64_t need = ralenet_conv1d_slab_bytes(a->B, a->Cin, a->Cout, a->K);
  RL_REQUIRE(slab_bytes >= need, RL_ERR_SHAPE, "conv1d_bwd_det: slab of %llu bytes, %llu needed",
             (unsigned long long)slab_bytes, (unsigned long long)need);
  const cudaStream_t st = (cudaStream_t)stream;
  RlDet det = {slab, (size_t)(slab_bytes / sizeof(float)), 0, {}, 0};
  rl_conv_bwd_args d = *a;                     // one partial slot per window (CTA)
  d.d_w = rl_det_take(&det, a->d_w, (size_t)a->Cout * a->Cin * a->K, a->B);
  d.d_b = a->d_w ? rl_det_take(&det, a->d_b, a->Cout, a->B) : nullptr;   // the kernels write d_b only with d_w
  RL_REQUIRE(rl_det_ok(&det), RL_ERR_SHAPE, "conv1d_bwd_det: slab too small");
  if (int rc = conv1d_bwd_launch<true>(&d, smem, st)) return rc;
  return rl_launch_grad_reduce(&det, st);
}

extern "C" int ralenet_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                            float beta2, float eps, int32_t step, float gscale, void* stream) {
  RL_REQUIRE(p && g && m && v, RL_ERR_NULL, "adam: NULL tensor");
  RL_REQUIRE(n > 0 && step >= 1, RL_ERR_SHAPE, "adam: n=%lld step=%d", (long long)n, step);
  RL_REQUIRE(((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16 == 0, RL_ERR_SHAPE,
             "adam: buffers must be 16-byte aligned");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2s = sqrtf(1.f - powf(beta2, (float)step));
  const int64_t nthreads = (n + 3) / 4;
  const int blocks = (int)((nthreads + RL_NT - 1) / RL_NT);
  rl_prof_pre((cudaStream_t)stream);
  adam_kernel<<<blocks, RL_NT, 0, (cudaStream_t)stream>>>(p, g, m, v, n, lr, beta1, beta2, eps, bc1, bc2s, gscale,
                                                          nullptr);
  return rl_check_launch("adam_kernel");
}

__global__ void step_inc_kernel(int32_t* s) { *s += 1; }

extern "C" int ralenet_adam_dev(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                                float beta2, float eps, int32_t* step_dev, float gscale, void* stream) {
  RL_REQUIRE(p && g && m && v && step_dev, RL_ERR_NULL, "adam_dev: NULL tensor");
  RL_REQUIRE(n > 0, RL_ERR_SHAPE, "adam_dev: n=%lld", (long long)n);
  RL_REQUIRE(((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16 == 0, RL_ERR_SHAPE,
             "adam_dev: buffers must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  rl_prof_pre(st);
  step_inc_kernel<<<1, 1, 0, st>>>(step_dev);
  if (int rc = rl_check_launch("step_inc_kernel")) return rc;
  const int64_t nthreads = (n + 3) / 4;
  const int blocks = (int)((nthreads + RL_NT - 1) / RL_NT);
  rl_prof_pre(st);
  adam_kernel<<<blocks, RL_NT, 0, st>>>(p, g, m, v, n, lr, beta1, beta2, eps, 1.f, 1.f, gscale, step_dev);
  return rl_check_launch("adam_kernel");
}
