// hg_abi.cu -- version, error reporting and device queries of the C ABI (include/hitgeom.h).
#include <stdarg.h>
#include <string.h>

#include "hg_common.cuh"

static thread_local char g_err[512] = "";

void hg_set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

unsigned long long g_hg_launches = 0;

HG_API int hg_version(void) { return 200; }

// Development knobs (benchmarks / A-B experiments only; not part of the stable ABI): small integer switches by name.
int g_hg_tune_knn_tc_off = 0;
HG_API int hg_tune(const char *key, int value) {
  if (key == nullptr) return HG_E_BADARG;
  if (!strcmp(key, "knn_tc")) {  // 1 = tensor-core kNN prefilter off (FP32 tile + row-select path)
    g_hg_tune_knn_tc_off = value;
    return HG_OK;
  }
  if (!strcmp(key, "small_fused")) {  // 1 = small clouds use the general (multi-kernel) finish / kNN-backward paths
    g_hg_tune_small_fused_off = value;
    return HG_OK;
  }
  // "prune" (0 = all-pairs kernels only, 1 = automatic), "prune_min_n" (size threshold, 0 = default), "prune_count"
  if (hg_prune_tune(key, value)) return HG_OK;
  hg_set_error("hg_tune: unknown key '%s'", key);
  return HG_E_BADARG;
}

HG_API unsigned long long hg_launch_count(void) { return g_hg_launches; }

HG_API const char *hg_last_error(void) { return g_err; }

int hg_sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

HG_API int hg_device_info(int *sm_count, int *clock_khz, long long *l2_bytes, long long *mem_bytes) {
  int dev = 0;
  HG_CUDA(cudaGetDevice(&dev));
  int v = 0;
  if (sm_count) {
    HG_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    *sm_count = v;
  }
  if (clock_khz) {
    HG_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrClockRate, dev));
    *clock_khz = v;
  }
  if (l2_bytes) {
    HG_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrL2CacheSize, dev));
    *l2_bytes = v;
  }
  if (mem_bytes) {
    size_t free_b = 0, total_b = 0;
    HG_CUDA(cudaMemGetInfo(&free_b, &total_b));
    *mem_bytes = (long long)total_b;
  }
  return HG_OK;
}

// ---- FP32 peak probe (bench.py's roofline denominator, next to the computed figure) ----------------------------------
// MEASURED_PEAKS.json carries no FP32 number, so the bench measures one: sixteen independent FFMA chains per thread
// (no memory traffic, full occupancy), 2 FLOP per FFMA, CUDA events around the launch.  Synchronises: call it outside
// timed regions.
namespace {
__global__ void __launch_bounds__(256) fp32_peak_kernel(float *__restrict__ out, int iters, float a, float b) {
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = (float)(threadIdx.x + i);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fmaf_rn(v[i], a, b);
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += v[i];
  if (s == 12345.678f) out[0] = s;  // (keeps the chains alive; never true in practice)
}
}  // namespace

HG_API int hg_probe_fp32_peak(float *tflops, float *scratch /*device, >= 4 bytes*/, hgStream stream_) {
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(tflops && scratch, HG_E_BADARG, "probe_fp32_peak: null pointer");
  const int iters = 8192, ctas = hg_sm_count() * 8;
  cudaEvent_t e0, e1;
  HG_CUDA(cudaEventCreate(&e0));
  HG_CUDA(cudaEventCreate(&e1));
  float best = 0.f;
  for (int rep = 0; rep < 4; ++rep) {  // the first launch warms the clocks up
    HG_CUDA(cudaEventRecord(e0, stream));
    fp32_peak_kernel<<<ctas, 256, 0, stream>>>(scratch, iters, 1.0000001f, 1e-9f);
    HG_CUDA(cudaEventRecord(e1, stream));
    HG_CUDA(cudaEventSynchronize(e1));
    float ms = 0.f;
    HG_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    const double flop = 2.0 * 16.0 * iters * 256.0 * ctas;
    if (rep > 0 && ms > 0.f) best = fmaxf(best, (float)(flop / (ms * 1e-3) / 1e12));
  }
  HG_CUDA(cudaEventDestroy(e0));
  HG_CUDA(cudaEventDestroy(e1));
  HG_CHECK_LAUNCH("fp32_peak_kernel");
  *tflops = best;
  return HG_OK;
}

// ---- optional per-kernel device timing (bench.py's roofline object) ---------------------------------------
// When enabled, the launch of each tagged hot kernel is bracketed by CUDA events recorded on the launching
// stream; hg_prof_read() returns the summed device time and the launch count.  Off by default (no events).
#include <vector>

namespace {
struct ProfTag {
  std::vector<cudaEvent_t> start, stop;
  int used = 0;
};
ProfTag g_prof[HG_PROF_NTAGS];
bool g_prof_on = false;
constexpr int kProfMaxPairs = 4096;
}  // namespace

bool hg_prof_begin(int tag, cudaStream_t s) {
  if (!g_prof_on || tag < 0 || tag >= HG_PROF_NTAGS) return false;
  ProfTag &t = g_prof[tag];
  if (t.used >= kProfMaxPairs) return false;
  if (t.used >= (int)t.start.size()) {
    cudaEvent_t a, b;
    if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return false;
    t.start.push_back(a);
    t.stop.push_back(b);
  }
  cudaEventRecord(t.start[t.used], s);
  return true;
}

void hg_prof_end(int tag, cudaStream_t s, bool began) {
  if (!began) return;
  ProfTag &t = g_prof[tag];
  cudaEventRecord(t.stop[t.used], s);
  t.used++;
}

HG_API void hg_prof_enable(int on) {
  g_prof_on = on != 0;
  for (int i = 0; i < HG_PROF_NTAGS; ++i) g_prof[i].used = 0;
}

HG_API int hg_prof_read(int tag, float *total_ms, int *launches) {
  HG_REQUIRE(tag >= 0 && tag < HG_PROF_NTAGS && total_ms && launches, HG_E_BADARG, "prof_read: bad tag");
  ProfTag &t = g_prof[tag];
  float sum = 0.f;
  for (int i = 0; i < t.used; ++i) {
    HG_CUDA(cudaEventSynchronize(t.stop[i]));
    float ms = 0.f;
    HG_CUDA(cudaEventElapsedTime(&ms, t.start[i], t.stop[i]));
    sum += ms;
  }
  *total_ms = sum;
  *launches = t.used;
  return HG_OK;
}
