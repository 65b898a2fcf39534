// synth.cu -- device-side training-batch synthesiser: the data path of SURVEY.md section 8 f3 with zero host traffic.
//
// The reference builds its training pairs on the host: wfdb records cut into 256-sample windows, z-normalised per lead
// (np_norm, local_utils/local_utils.py:261-266), real noise records (bw / ma / em) mixed in at a target SNR
// (Gnoisegen :86-114, single_snr_noise_add :176-192) and stored as .npy (data_utils.py:88-117), then fed through a
// DataLoader + collate (main.py:45-60).  None of that data ships, so benchmarks and tests use synthetic MIT-BIH-style
// windows (ecg_denoise_b200/synth.py, numpy).  This file is the same generator ON THE GPU -- beat trains of P-QRS-T
// Gaussians with the R peak of the middle beat at L/2 +- 8, per-lead z-normalisation, baseline-wander / muscle-artifact
// / electrode-motion style noise -- so that a training step can draw a fresh batch without touching the host:
//   ralenet_synth_windows  -> clean[B][leads][L], noise[B][leads][L]  (one CTA per window, counter-based RNG)
//   ralenet_snr_mix        -> noisy = clean + noise scaled to the target SNR (the reference's formula, eca.cu)
// The random stream is a pure function of (seed, *counter_dev, window, lead, sample): the same arguments give the same
// batch (CUDA-graph replays advance through *counter_dev, which the Adam step increments).  The numpy generator uses
// numpy's RandomState, so the two produce different (equally distributed) windows; what is checked is the definition:
// z-normalised leads, centred R peak, zero-mean noise, requested SNR.
#define RL_NT 256
#include "common.cuh"

namespace {

constexpr float FS = 360.f, TWO_PI = 6.283185307179586f;

struct Rng {
  uint64_t base;
  __device__ __forceinline__ float u01(uint32_t stream, uint32_t idx) const {        // (0, 1)
    const uint64_t h = mix64(base ^ mix64(((uint64_t)stream << 32) | idx));
    return ((float)(h >> 40) + 0.5f) * (1.0f / 16777216.0f);
  }
  __device__ __forceinline__ float normal(uint32_t stream, uint32_t idx) const {
    const float u1 = u01(stream, 2 * idx), u2 = u01(stream, 2 * idx + 1);
    return sqrtf(-2.f * __logf(u1)) * __cosf(TWO_PI * u2);
  }
};

// P-QRS-T complex: (offset s, width s, amplitude) relative to the R time -- the same five waves as synth.py::_beat
__constant__ float c_wave[5][3] = {{-0.20f, 0.025f, 0.12f}, {-0.035f, 0.010f, -0.14f}, {0.0f, 0.011f, 1.0f},
                                   {0.035f, 0.012f, -0.22f}, {0.25f, 0.055f, 0.30f}};

__device__ __forceinline__ float block_sum(float v, float* s_red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int w = 0; w < RL_NT / 32; ++w) r += s_red[w];
  return r;
}

// kind: 0 = bw, 1 = ma, 2 = em, 3 = emb (all three)
__global__ void __launch_bounds__(RL_NT) synth_windows_kernel(float* __restrict__ clean, float* __restrict__ noise, int B,
                                                             int leads, int L, uint64_t seed,
                                                             const int32_t* __restrict__ counter_dev, int kind) {
  __shared__ float s_red[RL_NT / 32];
  __shared__ float s_scan[2][1024];
  const int w = blockIdx.x, tid = threadIdx.x;
  const uint64_t ctr = counter_dev ? (uint64_t)(uint32_t)(*counter_dev) : 0ull;
  Rng rng{mix64(seed ^ mix64(ctr * 0x100000001b3ull + (uint64_t)w))};
  // window-level draws (every thread computes the same values)
  const float r_mid = (0.5f * L + floorf(rng.u01(0, 0) * 17.f) - 8.f) / FS;
  const float rr = 0.6f + 0.6f * rng.u01(0, 1);
  float r_time[7], amp_j[7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    r_time[k] = r_mid + (float)(k - 3) * rr * (1.f + 0.03f * rng.normal(1, k));
    amp_j[k] = 1.f + 0.1f * rng.normal(2, k);
  }
  for (int l = 0; l < leads; ++l) {
    const float gain = l == 0 ? 1.f : (0.4f + 0.5f * rng.u01(3, 2 * l)) * (rng.u01(3, 2 * l + 1) < 0.5f ? -1.f : 1.f);
    // ---- clean lead: beat train, then z-normalisation (np_norm: population std)
    float v[4];                                   // up to 4 samples per thread (L <= 1024)
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int t = tid + j * RL_NT;
      v[j] = 0.f;
      if (t < L) {
        const float ts = (float)t / FS;
        float y = 0.f;
#pragma unroll
        for (int k = 0; k < 7; ++k) {
          float b = 0.f;
#pragma unroll
          for (int q = 0; q < 5; ++q) {
            const float d = (ts - r_time[k] - c_wave[q][0]) / c_wave[q][1];
            b += c_wave[q][2] * __expf(-0.5f * d * d);
          }
          y += gain * amp_j[k] * b;
        }
        v[j] = y;
        sum += y;
      }
    }
    const float mean = block_sum(sum, s_red) / (float)L;
    float sq = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (tid + j * RL_NT < L) sq += (v[j] - mean) * (v[j] - mean);
    const float rstd = 1.f / (sqrtf(block_sum(sq, s_red) / (float)L) + 1e-8f);
    float* cw = clean + ((size_t)w * leads + l) * L;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (tid + j * RL_NT < L) cw[tid + j * RL_NT] = (v[j] - mean) * rstd;

    // ---- noise lead
    float nz[4] = {0.f, 0.f, 0.f, 0.f};
    if (kind == 0 || kind == 3) {                 // baseline wander: three slow sinusoids
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const float f = 0.05f + 0.45f * rng.u01(4 + l, 3 * s), ph = TWO_PI * rng.u01(4 + l, 3 * s + 1);
        const float am = 0.3f + 0.7f * rng.u01(4 + l, 3 * s + 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) nz[j] += am * __sinf(TWO_PI * f * (float)(tid + j * RL_NT) / FS + ph);
      }
    }
    if (kind == 1 || kind == 3) {                 // muscle artifact: white noise minus 0.7 x its 9-tap Hann smoothing
      const float hann[9] = {0.f, 0.036612f, 0.125f, 0.213388f, 0.25f, 0.213388f, 0.125f, 0.036612f, 0.f};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int t = tid + j * RL_NT;
        float sm = 0.f;
#pragma unroll
        for (int q = 1; q < 8; ++q) {
          const int tt = t + q - 4;
          if (tt >= 0 && tt < L) sm += hann[q] * rng.normal(16 + l, tt);
        }
        nz[j] += rng.normal(16 + l, t) - 0.7f * sm;
      }
    }
    if (kind == 2 || kind == 3) {                 // electrode motion: random walk of sparse steps + a little white noise
      for (int j = 0; j < 4; ++j) {
        const int t = tid + j * RL_NT;
        s_scan[0][t] = (t < L && rng.u01(32 + l, t) < 0.05f) ? rng.normal(40 + l, t) : 0.f;
      }
      __syncthreads();
      int cur = 0;
      for (int off = 1; off < 1024; off <<= 1) {   // Hillis-Steele inclusive scan over 1024 slots
        for (int j = 0; j < 4; ++j) {
          const int t = tid + j * RL_NT;
          s_scan[cur ^ 1][t] = s_scan[cur][t] + (t >= off ? s_scan[cur][t - off] : 0.f);
        }
        cur ^= 1;
        __syncthreads();
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int t = tid + j * RL_NT;
        nz[j] += s_scan[cur][t] + 0.05f * rng.normal(48 + l, t);
      }
      __syncthreads();
    }
    float ns = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (tid + j * RL_NT < L) ns += nz[j];
    const float nmean = block_sum(ns, s_red) / (float)L;
    float* nw = noise + ((size_t)w * leads + l) * L;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (tid + j * RL_NT < L) nw[tid + j * RL_NT] = nz[j] - nmean;
  }
}

}  // namespace

extern "C" int ralenet_synth_windows(float* clean, float* noise, int32_t B, int32_t leads, int32_t L, uint64_t seed,
                                     const int32_t* counter_dev, int32_t kind, void* stream) {
  RL_REQUIRE(clean && noise, RL_ERR_NULL, "synth_windows: NULL tensor");
  RL_REQUIRE(B > 0 && leads > 0 && leads <= 12 && L > 0 && L <= 1024 && kind >= 0 && kind <= 3, RL_ERR_SHAPE,
             "synth_windows: B=%d leads=%d L=%d kind=%d", B, leads, L, kind);
  rl_prof_pre((cudaStream_t)stream);
  synth_windows_kernel<<<B, RL_NT, 0, (cudaStream_t)stream>>>(clean, noise, B, leads, L, seed, counter_dev, kind);
  return rl_check_launch("synth_windows_kernel");
}
