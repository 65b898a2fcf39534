// api.cu -- error reporting, device check, launch accounting for libralenet_b200.so
#include <stdarg.h>
#include <string.h>
#include <atomic>
#include "common.cuh"

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};   // process-wide: backward runs on autograd threads

void rl_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

void rl_count_launch() { ++g_launches; }

// ---- optional per-launch timing (bench.py's roofline pass): one event after every launch on the
// profiled stream; a kernel's duration is the gap to the previous event (launches are serialised).
namespace {
constexpr int kMaxProf = 8192;
struct Prof {
  bool on = false;
  cudaStream_t stream = nullptr;
  int n = 0;
  cudaEvent_t ev[kMaxProf + 1];
  cudaEvent_t pre[kMaxProf];       // optional event right before a launch (excludes host-side gaps)
  bool has_pre[kMaxProf];
  int created = 0;
  char label[kMaxProf][48];
};
Prof g_prof;
}  // namespace

bool rl_prof_active() { return g_prof.on; }

void rl_prof_pre(cudaStream_t st) {
  if (g_prof.on && g_prof.n < kMaxProf && st == g_prof.stream) {
    cudaEventRecord(g_prof.pre[g_prof.n], st);
    g_prof.has_pre[g_prof.n] = true;
  }
}

int rl_check_launch(const char* what, int t0, int t1, const char* suffix) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    rl_set_error("%s: %s", what, cudaGetErrorString(e));
    return RL_ERR_CUDA;
  }
  ++g_launches;
  if (g_prof.on && g_prof.n < kMaxProf) {
    const int i = g_prof.n++;
    if (t1 >= 0) snprintf(g_prof.label[i], sizeof(g_prof.label[i]), "%s<%d,%d>%s", what, t0, t1, suffix);
    else if (t0 >= 0) snprintf(g_prof.label[i], sizeof(g_prof.label[i]), "%s<%d>%s", what, t0, suffix);
    else snprintf(g_prof.label[i], sizeof(g_prof.label[i]), "%s%s", what, suffix);
    cudaEventRecord(g_prof.ev[i + 1], g_prof.stream);
  }
  return RL_OK;
}

extern "C" int ralenet_profile_begin(void* stream) {
  while (g_prof.created <= kMaxProf) {
    if (g_prof.created < kMaxProf && cudaEventCreate(&g_prof.pre[g_prof.created]) != cudaSuccess) {
      rl_set_error("profile_begin: cudaEventCreate failed");
      return RL_ERR_CUDA;
    }
    if (cudaEventCreate(&g_prof.ev[g_prof.created]) != cudaSuccess) {
      rl_set_error("profile_begin: cudaEventCreate failed");
      return RL_ERR_CUDA;
    }
    ++g_prof.created;
  }
  g_prof.stream = (cudaStream_t)stream;
  g_prof.n = 0;
  for (int i = 0; i < kMaxProf; ++i) g_prof.has_pre[i] = false;
  g_prof.on = true;
  cudaEventRecord(g_prof.ev[0], g_prof.stream);
  return RL_OK;
}

extern "C" int ralenet_profile_end(char* labels, int32_t label_stride, float* ms, int32_t max_n) {
  g_prof.on = false;
  const int n = g_prof.n < max_n ? g_prof.n : max_n;
  if (g_prof.n > 0 && cudaEventSynchronize(g_prof.ev[g_prof.n]) != cudaSuccess) {
    rl_set_error("profile_end: cudaEventSynchronize failed");
    return RL_ERR_CUDA;
  }
  for (int i = 0; i < n; ++i) {
    cudaEventElapsedTime(&ms[i], g_prof.has_pre[i] ? g_prof.pre[i] : g_prof.ev[i], g_prof.ev[i + 1]);
    snprintf(labels + (size_t)i * label_stride, label_stride, "%s", g_prof.label[i]);
  }
  return n;
}

extern "C" int ralenet_abi_version(void) { return RL_ABI_VERSION; }
extern "C" const char* ralenet_last_error(void) { return g_err; }

extern "C" int ralenet_check_device(int dev) {
  cudaDeviceProp p;
  cudaError_t e = cudaGetDeviceProperties(&p, dev);
  if (e != cudaSuccess) {
    rl_set_error("cudaGetDeviceProperties(%d): %s", dev, cudaGetErrorString(e));
    return RL_ERR_CUDA;
  }
  if (p.major != 10) {
    rl_set_error("device %d is sm_%d%d; libralenet_b200 is built for sm_100a only (no fallback path)", dev, p.major,
                 p.minor);
    return RL_ERR_ARCH;
  }
  return RL_OK;
}

extern "C" int64_t ralenet_launch_count(int32_t reset) {
  return reset ? g_launches.exchange(0) : g_launches.load();
}
