// records.cu -- record <-> window pipeline around the network for long recordings (inference, SURVEY.md 8f-2).
//
// The reference cuts 2-lead records into 256-sample windows on the host with numpy
// (local_utils/local_utils.py:47-65, 116-130) after per-lead z-normalisation (np_norm, :261-266) and never
// stitches them back.  Here: per-(record, lead) statistics, a fused z-norm + window gather, and a
// deterministic overlap-add stitch (gather form, no atomics) that also undoes the normalisation.
// All three are HBM-bound streaming kernels.
// For training (SURVEY.md 8f-3), record_sample_kernel draws the same z-normalised windows from a record bank in a
// keyed per-epoch order and pairs each with a window of a noise bank and an SNR level; ralenet_snr_mix does the mix.
// For evaluation, record_enumerate_kernel walks every (grid window, level) pair of held-out banks once, in order,
// with a noise pick fixed per pair.
#include "common.cuh"

namespace {

// one CTA per (record, lead): mean and 1/std (population std, like numpy's default in np_norm)
__global__ void __launch_bounds__(RL_NT) record_stats_kernel(const float* __restrict__ x, int64_t T,
                                                             float* __restrict__ stats) {
  __shared__ double sd[2 * (RL_NT / 32)];
  const float* xr = x + (size_t)blockIdx.x * T;
  double s = 0.0, q = 0.0;
  for (int64_t i = threadIdx.x; i < T; i += RL_NT) {
    const double v = (double)__ldg(xr + i);
    s += v;
    q += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) { sd[2 * w] = s; sd[2 * w + 1] = q; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ts = 0.0, tq = 0.0;
    for (int k = 0; k < RL_NT / 32; ++k) { ts += sd[2 * k]; tq += sd[2 * k + 1]; }
    const double mean = ts / (double)T;
    const double var = fmax(tq / (double)T - mean * mean, 0.0);
    stats[2 * blockIdx.x] = (float)mean;
    stats[2 * blockIdx.x + 1] = (float)(1.0 / sqrt(var + 1e-12));
  }
}

// win[(r*nper + w)][c][i] = (x[r][c][w*stride + i] - mean[r][c]) * rstd[r][c]
__global__ void __launch_bounds__(RL_NT) window_gather_kernel(const float* __restrict__ x, const float* __restrict__ stats,
                                                              float* __restrict__ win, int C, int64_t T, int W,
                                                              int stride, int nper, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * RL_NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * RL_NT) {
    const int i = (int)(idx % W);
    const int64_t rest = idx / W;
    const int c = (int)(rest % C);
    const int64_t wg = rest / C;                 // global window index
    const int w = (int)(wg % nper);
    const int64_t r = wg / nper;
    const size_t rc = (size_t)r * C + c;
    float v = __ldg(x + rc * T + (int64_t)w * stride + i);
    if (stats) v = (v - __ldg(stats + 2 * rc)) * __ldg(stats + 2 * rc + 1);
    win[idx] = v;
  }
}

// y[r][c][t] = mean over the windows covering t of win[...][c][t - w*stride], de-normalised; samples not covered
// by any full window pass the input through unchanged.
__global__ void __launch_bounds__(RL_NT) window_scatter_kernel(const float* __restrict__ win,
                                                               const float* __restrict__ x,
                                                               const float* __restrict__ stats, float* __restrict__ y,
                                                               int C, int64_t T, int W, int stride, int nper,
                                                               int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * RL_NT + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * RL_NT) {
    const int64_t t = idx % T;
    const size_t rc = (size_t)(idx / T);
    const int c = (int)(rc % C);
    const int64_t r = (int64_t)(rc / C);
    int64_t w_hi = t / stride;
    if (w_hi > nper - 1) w_hi = nper - 1;
    int64_t w_lo = (t - W + stride) / stride;    // ceil((t - W + 1) / stride) for t - W + 1 >= 0
    if (t - W + 1 <= 0) w_lo = 0;
    float s = 0.f;
    int n = 0;
    for (int64_t w = w_lo; w <= w_hi; ++w) {
      const int64_t off = t - w * stride;
      if (off >= 0 && off < W) {
        s += __ldg(win + (((size_t)(r * nper + w)) * C + c) * W + off);
        ++n;
      }
    }
    float out;
    if (n > 0) {
      out = s / (float)n;
      if (stats) out = out / __ldg(stats + 2 * rc + 1) + __ldg(stats + 2 * rc);
    } else {
      out = __ldg(x + idx);
    }
    y[idx] = out;
  }
}

// ---- training-window sampler: the reference's data recipe (cut, np_norm, noise at a target SNR) drawn on the device
constexpr int FEISTEL_ROUNDS = 4;

// keyed bijection of [0, n): a balanced Feistel network on the smallest even bit width 2h >= 2 with 2^(2h) >= n,
// walked until the value falls back into [0, n) (the walk ends because x itself lies on a cycle that enters [0, n))
__device__ __forceinline__ uint64_t feistel_perm(uint64_t x, uint64_t n, uint64_t key) {
  int h = 1;
  while ((1ull << (2 * h)) < n) ++h;
  const uint64_t m = (1ull << h) - 1;
  do {
    uint64_t l = x >> h, r = x & m;
#pragma unroll
    for (int k = 0; k < FEISTEL_ROUNDS; ++k) {
      const uint64_t t = l ^ (mix64(r ^ mix64(key + k)) & m);
      l = r;
      r = t;
    }
    x = (l << h) | r;
  } while (x >= n);
  return x;
}

// Slot i of a drawn batch <- clean window (rec, off) of the record bank, z-normalised with the arithmetic of
// window_gather_kernel, and noise window (nrec, noff) of the noise bank; clean lead l reads noise lead l % noise_leads.
// A is rl_sample_args or rl_enum_args (same bank fields).
template <typename A>
__device__ __forceinline__ void copy_window_pair(const A& a, int i, int tid, int W, int64_t rec, int64_t off,
                                                 int64_t nrec, int64_t noff) {
  for (int l = 0; l < a.leads; ++l) {
    const size_t rc = (size_t)rec * a.leads + l;
    const float* xs = a.records + rc * a.T + off;
    const float* ns = a.noise + ((size_t)nrec * a.noise_leads + l % a.noise_leads) * a.Tn + noff;
    float mean = 0.f, rstd = 1.f;
    if (a.stats) { mean = __ldg(a.stats + 2 * rc); rstd = __ldg(a.stats + 2 * rc + 1); }
    float* cw = a.clean_out + ((size_t)i * a.leads + l) * W;
    float* nw = a.noise_out + ((size_t)i * a.leads + l) * W;
    for (int t = tid; t < W; t += RL_NT) {
      float v = __ldg(xs + t);
      const float nz = __ldg(ns + t);
      if (a.stats) v = (v - mean) * rstd;          // the arithmetic of window_gather_kernel
      cw[t] = v;
      nw[t] = nz;
    }
  }
}

// one CTA per window; the plan (which record window, which noise window, which SNR level) is computed by every thread
__global__ void __launch_bounds__(RL_NT) record_sample_kernel(rl_sample_args a, int nper, uint64_t n, uint64_t spe) {
  pdl_wait();                                     // *counter may be the Adam step counter the previous kernel bumped
  pdl_trigger();
  const int i = blockIdx.x, tid = threadIdx.x, W = a.W;
  const uint64_t ctr = a.counter ? (uint64_t)(uint32_t)(*a.counter) : 0ull;
  const uint64_t slot = (uint64_t)a.rank * a.B + i;                        // slot within the world batch
  const uint64_t g = (ctr % spe) * (uint64_t)a.world * a.B + slot;         // position in this epoch's order
  const uint64_t item = feistel_perm(g, n, mix64(a.seed ^ mix64(2 * (ctr / spe))));
  const int64_t rec = (int64_t)(item / nper), off = (int64_t)(item % nper) * a.stride;
  const uint64_t hw = mix64(mix64(a.seed ^ mix64(2 * ctr + 1)) ^ slot);
  const int64_t nrec = (int64_t)(mix64(hw + 1) % (uint64_t)a.N);
  const int64_t noff = (int64_t)(mix64(hw + 2) % (uint64_t)(a.Tn - W + 1));
  const int lvl = (int)(mix64(hw + 3) % (uint64_t)a.n_snr);
  if (tid == 0) {
    a.snr_out[i] = __ldg(a.snr_levels + lvl);
    if (a.meta) {
      a.meta[4 * i] = (int32_t)rec;
      a.meta[4 * i + 1] = (int32_t)off;
      a.meta[4 * i + 2] = (int32_t)nrec;
      a.meta[4 * i + 3] = (int32_t)noff;
    }
  }
  copy_window_pair(a, i, tid, W, rec, off, nrec, noff);
}

// one CTA per slot of the ordered evaluation draw: item e = g * n_snr + lvl of the (grid window, level) set, in
// order; the noise pick hashes (seed, g, lvl) only.  Slots past the end of the set are zero-filled and marked -1.
__global__ void __launch_bounds__(RL_NT) record_enumerate_kernel(rl_enum_args a, int nper, uint64_t n_eval) {
  pdl_wait();                                     // *counter may have been bumped by the previous eval_reduce_kernel
  pdl_trigger();
  const int i = blockIdx.x, tid = threadIdx.x, W = a.W;
  const uint64_t ctr = a.counter ? (uint64_t)(uint32_t)(*a.counter) : 0ull;
  const uint64_t e = ctr * (uint64_t)a.world * a.B + (uint64_t)a.rank * a.B + i;
  if (e >= n_eval) {
    if (tid == 0) {
      a.snr_out[i] = 0.f;
      a.level[i] = -1;
      if (a.meta)
        for (int k = 0; k < 4; ++k) a.meta[4 * i + k] = -1;
    }
    const size_t per = (size_t)a.leads * W;
    for (size_t t = tid; t < per; t += RL_NT) {
      a.clean_out[i * per + t] = 0.f;
      a.noise_out[i * per + t] = 0.f;
    }
    return;
  }
  const uint64_t g = e / (uint64_t)a.n_snr;
  const int lvl = (int)(e % (uint64_t)a.n_snr);
  const int64_t rec = (int64_t)(g / nper), off = (int64_t)(g % nper) * a.stride;
  const uint64_t hw = mix64(mix64(a.seed ^ mix64(g)) ^ (uint64_t)lvl);
  const int64_t nrec = (int64_t)(mix64(hw + 1) % (uint64_t)a.N);
  const int64_t noff = (int64_t)(mix64(hw + 2) % (uint64_t)(a.Tn - W + 1));
  if (tid == 0) {
    a.snr_out[i] = __ldg(a.snr_levels + lvl);
    a.level[i] = lvl;
    if (a.meta) {
      a.meta[4 * i] = (int32_t)rec;
      a.meta[4 * i + 1] = (int32_t)off;
      a.meta[4 * i + 2] = (int32_t)nrec;
      a.meta[4 * i + 3] = (int32_t)noff;
    }
  }
  copy_window_pair(a, i, tid, W, rec, off, nrec, noff);
}

}  // namespace

extern "C" int ralenet_record_stats(const float* x, int32_t RC, int64_t T, float* stats, void* stream) {
  RL_REQUIRE(x && stats, RL_ERR_NULL, "record_stats: NULL tensor");
  RL_REQUIRE(RC > 0 && T > 0, RL_ERR_SHAPE, "record_stats: RC=%d T=%lld", RC, (long long)T);
  record_stats_kernel<<<RC, RL_NT, 0, (cudaStream_t)stream>>>(x, T, stats);
  return rl_check_launch("record_stats_kernel");
}

static int rec_check(int32_t R, int32_t C, int64_t T, int32_t W, int32_t stride, int32_t* nper) {
  RL_REQUIRE(R > 0 && C > 0 && T >= W && W > 0 && stride > 0 && stride <= W, RL_ERR_SHAPE,
             "records: unsupported R=%d C=%d T=%lld W=%d stride=%d", R, C, (long long)T, W, stride);
  *nper = (int32_t)((T - W) / stride + 1);
  return RL_OK;
}

extern "C" int32_t ralenet_windows_per_record(int64_t T, int32_t W, int32_t stride) {
  if (T < W || W <= 0 || stride <= 0) return 0;
  return (int32_t)((T - W) / stride + 1);
}

extern "C" int ralenet_window_gather(const float* x, const float* stats, float* win, int32_t R, int32_t C, int64_t T,
                                     int32_t W, int32_t stride, void* stream) {
  RL_REQUIRE(x && win, RL_ERR_NULL, "window_gather: NULL tensor");
  int32_t nper = 0;
  if (int rc = rec_check(R, C, T, W, stride, &nper)) return rc;
  const int64_t total = (int64_t)R * nper * C * W;
  const int blocks = (int)((total + RL_NT * 4 - 1) / (RL_NT * 4) < 148 * 32 ? (total + RL_NT * 4 - 1) / (RL_NT * 4) : 148 * 32);
  window_gather_kernel<<<blocks < 1 ? 1 : blocks, RL_NT, 0, (cudaStream_t)stream>>>(x, stats, win, C, T, W, stride, nper,
                                                                                    total);
  return rl_check_launch("window_gather_kernel");
}

extern "C" int ralenet_window_scatter(const float* win, const float* x, const float* stats, float* y, int32_t R,
                                      int32_t C, int64_t T, int32_t W, int32_t stride, void* stream) {
  RL_REQUIRE(win && x && y, RL_ERR_NULL, "window_scatter: NULL tensor");
  int32_t nper = 0;
  if (int rc = rec_check(R, C, T, W, stride, &nper)) return rc;
  const int64_t total = (int64_t)R * C * T;
  const int blocks = (int)((total + RL_NT * 4 - 1) / (RL_NT * 4) < 148 * 32 ? (total + RL_NT * 4 - 1) / (RL_NT * 4) : 148 * 32);
  window_scatter_kernel<<<blocks < 1 ? 1 : blocks, RL_NT, 0, (cudaStream_t)stream>>>(win, x, stats, y, C, T, W, stride,
                                                                                     nper, total);
  return rl_check_launch("window_scatter_kernel");
}

extern "C" int ralenet_record_sample(const rl_sample_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "record_sample: args is NULL");
  RL_REQUIRE(a->records && a->noise && a->snr_levels && a->clean_out && a->noise_out && a->snr_out, RL_ERR_NULL,
             "record_sample: NULL tensor");
  RL_REQUIRE(a->R > 0 && a->leads > 0 && a->leads <= 12 && a->N > 0 && a->B > 0 && a->W > 0 && a->stride > 0 &&
                 a->n_snr >= 1 && a->W <= a->T && a->W <= a->Tn,
             RL_ERR_SHAPE, "record_sample: unsupported R=%d leads=%d T=%lld N=%d Tn=%lld W=%d stride=%d B=%d n_snr=%d",
             a->R, a->leads, (long long)a->T, a->N, (long long)a->Tn, a->W, a->stride, a->B, a->n_snr);
  RL_REQUIRE(a->noise_leads == 1 || a->noise_leads == a->leads, RL_ERR_SHAPE,
             "record_sample: noise_leads=%d must be 1 or leads=%d", a->noise_leads, a->leads);
  RL_REQUIRE(a->world > 0 && a->rank >= 0 && a->rank < a->world, RL_ERR_SHAPE, "record_sample: rank=%d world=%d",
             a->rank, a->world);
  RL_REQUIRE(!a->meta || (a->T <= INT32_MAX && a->Tn <= INT32_MAX), RL_ERR_SHAPE,
             "record_sample: meta holds int32 offsets; T=%lld Tn=%lld", (long long)a->T, (long long)a->Tn);
  const int64_t nper = (a->T - a->W) / a->stride + 1;
  RL_REQUIRE(nper <= INT32_MAX, RL_ERR_SHAPE, "record_sample: %lld windows per record", (long long)nper);
  const uint64_t n = (uint64_t)a->R * (uint64_t)nper, spe = n / ((uint64_t)a->world * (uint64_t)a->B);
  RL_REQUIRE(spe > 0, RL_ERR_SHAPE, "record_sample: %llu grid windows are fewer than world*B=%lld",
             (unsigned long long)n, (long long)a->world * a->B);
  rl_launch_pdl(record_sample_kernel, dim3(a->B), dim3(RL_NT), 0, (cudaStream_t)stream, *a, (int)nper, n, spe);
  return rl_check_launch("record_sample_kernel");
}

extern "C" int ralenet_record_enumerate(const rl_enum_args* a, void* stream) {
  RL_REQUIRE(a, RL_ERR_NULL, "record_enumerate: args is NULL");
  RL_REQUIRE(a->records && a->noise && a->snr_levels && a->clean_out && a->noise_out && a->snr_out && a->level,
             RL_ERR_NULL, "record_enumerate: NULL tensor");
  RL_REQUIRE(a->R > 0 && a->leads > 0 && a->leads <= 12 && a->N > 0 && a->B > 0 && a->W > 0 && a->stride > 0 &&
                 a->n_snr >= 1 && a->W <= a->T && a->W <= a->Tn,
             RL_ERR_SHAPE,
             "record_enumerate: unsupported R=%d leads=%d T=%lld N=%d Tn=%lld W=%d stride=%d B=%d n_snr=%d", a->R,
             a->leads, (long long)a->T, a->N, (long long)a->Tn, a->W, a->stride, a->B, a->n_snr);
  RL_REQUIRE(a->noise_leads == 1 || a->noise_leads == a->leads, RL_ERR_SHAPE,
             "record_enumerate: noise_leads=%d must be 1 or leads=%d", a->noise_leads, a->leads);
  RL_REQUIRE(a->world > 0 && a->rank >= 0 && a->rank < a->world, RL_ERR_SHAPE, "record_enumerate: rank=%d world=%d",
             a->rank, a->world);
  RL_REQUIRE(a->T <= INT32_MAX && a->Tn <= INT32_MAX, RL_ERR_SHAPE,
             "record_enumerate: offsets are int32; T=%lld Tn=%lld", (long long)a->T, (long long)a->Tn);
  const int64_t nper = (a->T - a->W) / a->stride + 1;
  const uint64_t grid = (uint64_t)a->R * (uint64_t)nper;                              // < 2^62
  RL_REQUIRE(grid <= (1ull << 62) / (uint64_t)a->n_snr, RL_ERR_SHAPE,
             "record_enumerate: %llu grid windows x %d levels overflow the item index", (unsigned long long)grid,
             a->n_snr);
  const uint64_t n_eval = grid * (uint64_t)a->n_snr;
  rl_launch_pdl(record_enumerate_kernel, dim3(a->B), dim3(RL_NT), 0, (cudaStream_t)stream, *a, (int)nper, n_eval);
  return rl_check_launch("record_enumerate_kernel");
}
