// hg_host.cu -- the CW-kNN distance step on HOST buffers (the end-to-end entry point of the C ABI).
//
// One call = what a CW-kNN attack iteration asks of the distance term (CW/kNN.py:104-108 with
// util/dist_utils.py:258-294 ChamferkNNDist, batch_avg=True): adversarial and original clouds in host memory ->
// loss (host scalar) and d loss / d adv (host array).  The batch is cut into chunks of clouds (clouds are
// independent, SURVEY.md section 8e) that go through two sets of device buffers: all kernels run back to back on ONE
// compute stream (kernels of two chunks on two streams only contend: 117.3 -> 116.4 ms per config-5 step), the copies of
// a buffer set on its own stream, events in between: while chunk i computes, chunk i+1 is copied in and the gradient of
// chunk i-1 is copied out, so PCIe/NVLink-C2C traffic disappears behind the kernels instead of adding to them.  The kernels are the same entry points the
// device-pointer ABI exposes (hg_nn_bidir_f32, hg_set_loss_*, hg_knn_self_f32, hg_knn_outlier_*): results are
// bit-identical to calling those on a resident batch.
#include <new>
#include <vector>

#include "hg_common.cuh"

struct hgHostStep {
  int N = 0, chunk = 0, k1max = 0, device = 0;
  float *loss_pinned = nullptr;  // [loss_cap] page-locked staging for the per-cloud losses: a D2H copy into pageable
  int loss_cap = 0;              // memory would block the host inside the loop and serialise the pipeline
  cudaStream_t compute = nullptr;  // all kernels, back to back (two streams of kernels would only contend)
  struct Slot {
    cudaStream_t stream = nullptr;   // this slot's copies, both directions
    cudaEvent_t done = nullptr;      // (unused) D2H of the previous use of this slot finished
    cudaEvent_t in_ready = nullptr;  // this slot's host-to-device copies have landed
    cudaEvent_t comp_done = nullptr; // this slot's kernels have finished
    float *adv = nullptr, *ori = nullptr, *grad_ch = nullptr, *grad_knn = nullptr;
    float *min1 = nullptr, *min2 = nullptr, *vals = nullptr, *value = nullptr, *mask = nullptr;
    int *arg1 = nullptr, *arg2 = nullptr, *idx = nullptr;
    float *loss1 = nullptr, *loss2 = nullptr, *lossk = nullptr, *w = nullptr, *g1 = nullptr, *g2 = nullptr,
          *gk = nullptr, *total = nullptr;
    void *ws = nullptr;
    size_t ws_bytes = 0;
  } slot[2];
};

namespace {

// the session's buffers and streams live on the device that was current at creation: calls run there whatever the
// caller's current device is, and put it back afterwards
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

// per cloud: total = w (cw * pick(loss1, loss2) + kw * lossk); upstream scales of the three partial losses
__global__ void host_step_scales_kernel(const float *__restrict__ loss1, const float *__restrict__ loss2,
                                        const float *__restrict__ lossk, const float *__restrict__ w, int n, int method,
                                        float cw, float kw, float inv_b, float *__restrict__ g1,
                                        float *__restrict__ g2, float *__restrict__ gk, float *__restrict__ total) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float wi = w ? w[i] : 1.0f;
  const float ch = method == 0 ? loss1[i] : method == 1 ? loss2[i] : (loss1[i] + loss2[i]) / 2.0f;
  total[i] = __fadd_rn(__fmul_rn(__fmul_rn(ch, wi), cw), __fmul_rn(__fmul_rn(lossk[i], wi), kw));
  const float gc = __fmul_rn(__fmul_rn(cw, inv_b), wi);
  g1[i] = method == 0 ? gc : method == 1 ? 0.f : gc / 2.0f;
  g2[i] = method == 1 ? gc : method == 0 ? 0.f : gc / 2.0f;
  gk[i] = __fmul_rn(__fmul_rn(kw, inv_b), wi);
}

__global__ void __launch_bounds__(256) host_step_add_kernel(float *__restrict__ a, const float *__restrict__ b,
                                                            long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    a[i] = __fadd_rn(a[i], b[i]);
}

template <typename T>
int dev_alloc(T **p, size_t count) {
  HG_CUDA(cudaMalloc((void **)p, count * sizeof(T)));
  return HG_OK;
}

size_t slot_workspace_bytes(int chunk, int N, int k1) {
  size_t a = hg_nn_bidir_workspace_bytes(chunk, N, N, 3);
  size_t b = hg_set_loss_bwd_workspace_bytes(chunk, N, N);
  size_t c = hg_knn_self_workspace_bytes(chunk, N, 3, k1);
  size_t d = hg_knn_outlier_bwd_workspace_bytes(chunk, N, k1);
  size_t m = a > b ? a : b;
  m = m > c ? m : c;
  return m > d ? m : d;
}

void free_session(hgHostStep *s) {
  for (auto &sl : s->slot) {
    float *fp[] = {sl.adv, sl.ori, sl.grad_ch, sl.grad_knn, sl.min1, sl.min2, sl.vals, sl.value, sl.mask,
                   sl.loss1, sl.loss2, sl.lossk, sl.w, sl.g1, sl.g2, sl.gk, sl.total};
    for (float *p : fp)
      if (p) cudaFree(p);
    int *ip[] = {sl.arg1, sl.arg2, sl.idx};
    for (int *p : ip)
      if (p) cudaFree(p);
    if (sl.ws) cudaFree(sl.ws);
    if (sl.done) cudaEventDestroy(sl.done);
    if (sl.in_ready) cudaEventDestroy(sl.in_ready);
    if (sl.comp_done) cudaEventDestroy(sl.comp_done);
    if (sl.stream) cudaStreamDestroy(sl.stream);
  }
  if (s->compute) cudaStreamDestroy(s->compute);
  if (s->loss_pinned) cudaFreeHost(s->loss_pinned);
  delete s;
}

int init_session(hgHostStep *s) {
  const size_t pts = (size_t)s->chunk * s->N;
  HG_CUDA(cudaStreamCreateWithFlags(&s->compute, cudaStreamNonBlocking));
  for (auto &sl : s->slot) {
    HG_CUDA(cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking));
    HG_CUDA(cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming));
    HG_CUDA(cudaEventCreateWithFlags(&sl.in_ready, cudaEventDisableTiming));
    HG_CUDA(cudaEventCreateWithFlags(&sl.comp_done, cudaEventDisableTiming));
    int rc = 0;
    rc |= dev_alloc(&sl.adv, pts * 3) | dev_alloc(&sl.ori, pts * 3) | dev_alloc(&sl.grad_ch, pts * 3) |
          dev_alloc(&sl.grad_knn, pts * 3);
    rc |= dev_alloc(&sl.min1, pts) | dev_alloc(&sl.min2, pts) | dev_alloc(&sl.arg1, pts) | dev_alloc(&sl.arg2, pts);
    rc |= dev_alloc(&sl.vals, pts * s->k1max) | dev_alloc(&sl.idx, pts * s->k1max) | dev_alloc(&sl.value, pts) |
          dev_alloc(&sl.mask, pts);
    float **small[] = {&sl.loss1, &sl.loss2, &sl.lossk, &sl.w, &sl.g1, &sl.g2, &sl.gk, &sl.total};
    for (float **p : small) rc |= dev_alloc(p, (size_t)s->chunk);
    if (rc) return rc;
    sl.ws_bytes = slot_workspace_bytes(s->chunk, s->N, s->k1max);
    HG_CUDA(cudaMalloc(&sl.ws, sl.ws_bytes ? sl.ws_bytes : 256));
  }
  return HG_OK;
}

}  // namespace

HG_API hgHostStep *hg_host_step_create(int N, int chunk_clouds, int knn_k_max) {
  if (N <= 0 || chunk_clouds <= 0 || knn_k_max < 1 || knn_k_max + 1 > 32 || knn_k_max + 1 > N) {
    hg_set_error("host_step_create: need N > 0, chunk_clouds > 0, 1 <= knn_k_max <= min(31, N-1)");
    return nullptr;
  }
  hgHostStep *s = new (std::nothrow) hgHostStep();
  if (!s) return nullptr;
  s->N = N;
  s->chunk = chunk_clouds;
  s->k1max = knn_k_max + 1;
  cudaGetDevice(&s->device);
  if (init_session(s) != HG_OK) {
    free_session(s);
    return nullptr;
  }
  return s;
}

HG_API void hg_host_step_destroy(hgHostStep *s) {
  if (!s) return;
  DeviceGuard guard(s->device);
  free_session(s);
}

HG_API int hg_chamfer_knn_step_host_f32(hgHostStep *s, const float *adv_h, const float *ori_h, int B,
                                        int chamfer_method, int knn_k, float knn_alpha, float chamfer_weight,
                                        float knn_weight, const float *weights_h, float *loss_h,
                                        float *cloud_loss_h, float *grad_adv_h) {
  HG_NVTX_RANGE("hg_chamfer_knn_step_host_f32");
  HG_REQUIRE(s && adv_h && ori_h && loss_h && cloud_loss_h && grad_adv_h, HG_E_BADARG, "chamfer_knn_step_host: null pointer");
  HG_REQUIRE(B > 0, HG_E_BADARG, "chamfer_knn_step_host: B must be positive");
  HG_REQUIRE(chamfer_method >= 0 && chamfer_method <= 2, HG_E_BADARG, "chamfer_knn_step_host: method must be 0, 1 or 2");
  HG_REQUIRE(knn_k >= 1 && knn_k + 1 <= s->k1max, HG_E_BADARG, "chamfer_knn_step_host: knn_k=%d exceeds the session's %d",
             knn_k, s->k1max - 1);
  const int N = s->N, k1 = knn_k + 1;
  const float inv_b = 1.0f / (float)B;
  DeviceGuard guard(s->device);
  if (B > s->loss_cap) {
    if (s->loss_pinned) cudaFreeHost(s->loss_pinned);
    s->loss_pinned = nullptr;
    s->loss_cap = 0;
    HG_CUDA(cudaMallocHost((void **)&s->loss_pinned, (size_t)B * sizeof(float)));
    s->loss_cap = B;
  }
  // chunk schedule: short chunks at both ends -- the first chunk's host-to-device copy and the last chunk's
  // device-to-host copy are the only transfers nothing can hide behind -- full-size chunks in between (fewer launches
  // and kernel tails): 1024 clouds in slots of 256 go as 32, 96, 256, 256, 256, 96, 32 (116.5 -> 114.9 ms per step)
  std::vector<int> sched;
  {
    const int c = s->chunk, head[2] = {c / 8 > 0 ? c / 8 : 1, (3 * c) / 8 > 0 ? (3 * c) / 8 : 1};
    int left = B;
    if (B >= 2 * c) {
      for (int h = 0; h < 2; ++h) {
        sched.push_back(head[h]);
        left -= 2 * head[h];
      }
      while (left > 0) {
        const int nb = left < c ? left : c;
        sched.push_back(nb);
        left -= nb;
      }
      sched.push_back(head[1]);
      sched.push_back(head[0]);
    } else {
      while (left > 0) {
        const int nb = left < c ? left : c;
        sched.push_back(nb);
        left -= nb;
      }
    }
  }
  int use = 0, b0 = 0;
  for (size_t ci = 0; ci < sched.size(); b0 += sched[ci], ++ci, use ^= 1) {
    auto &sl = s->slot[use];
    const int nb = sched[ci];
    const size_t pts = (size_t)nb * N, off = (size_t)b0 * N * 3;
    // copies on the slot's stream, kernels on the one compute stream, events in between.  The slot stream's order
    // already guarantees that this slot's previous D2H finished before its buffers are rewritten.
    cudaStream_t cp = sl.stream, st = s->compute;
    hgStream hs = (hgStream)st;
    HG_CUDA(cudaMemcpyAsync(sl.adv, adv_h + off, pts * 3 * sizeof(float), cudaMemcpyHostToDevice, cp));
    HG_CUDA(cudaMemcpyAsync(sl.ori, ori_h + off, pts * 3 * sizeof(float), cudaMemcpyHostToDevice, cp));
    if (weights_h) HG_CUDA(cudaMemcpyAsync(sl.w, weights_h + b0, (size_t)nb * sizeof(float), cudaMemcpyHostToDevice, cp));
    HG_CUDA(cudaEventRecord(sl.in_ready, cp));
    HG_CUDA(cudaStreamWaitEvent(st, sl.in_ready, 0));
    int rc = hg_nn_bidir_f32(sl.ori, sl.adv, nb, N, N, 3, sl.min1, sl.arg1, sl.min2, sl.arg2, sl.ws, sl.ws_bytes, hs);
    if (rc) return rc;
    rc = hg_set_loss_f32(sl.min1, sl.min2, nb, N, N, HG_MODE_CHAMFER, sl.loss1, sl.loss2, nullptr, nullptr, hs);
    if (rc) return rc;
    rc = hg_knn_self_f32(sl.adv, nb, N, 3, k1, sl.vals, sl.idx, sl.ws, sl.ws_bytes, hs);
    if (rc) return rc;
    rc = hg_knn_outlier_fwd_f32(sl.vals, nb, N, k1, knn_alpha, nullptr, sl.value, sl.mask, sl.lossk, hs);
    if (rc) return rc;
    host_step_scales_kernel<<<(nb + 127) / 128, 128, 0, st>>>(sl.loss1, sl.loss2, sl.lossk, weights_h ? sl.w : nullptr, nb,
                                                              chamfer_method, chamfer_weight, knn_weight, inv_b, sl.g1,
                                                              sl.g2, sl.gk, sl.total);
    HG_CHECK_LAUNCH("host_step_scales_kernel");
    rc = hg_set_loss_bwd_f32(sl.ori, sl.adv, sl.arg1, sl.arg2, nullptr, nullptr, chamfer_method == 1 ? nullptr : sl.g1,
                             chamfer_method == 0 ? nullptr : sl.g2, nb, N, N, 3,
                             HG_MODE_CHAMFER, sl.grad_ch, nullptr, sl.ws, sl.ws_bytes, hs);
    if (rc) return rc;
    rc = hg_knn_outlier_bwd_f32(sl.adv, sl.idx, sl.mask, sl.gk, nb, N, 3, k1, sl.grad_knn, sl.ws, sl.ws_bytes, hs);
    if (rc) return rc;
    {
      const long long n = (long long)pts * 3;
      host_step_add_kernel<<<hg_grid_for(n, 256, 16), 256, 0, st>>>(sl.grad_ch, sl.grad_knn, n);
      HG_CHECK_LAUNCH("host_step_add_kernel");
    }
    HG_CUDA(cudaEventRecord(sl.comp_done, st));
    HG_CUDA(cudaStreamWaitEvent(cp, sl.comp_done, 0));
    HG_CUDA(cudaMemcpyAsync(grad_adv_h + off, sl.grad_ch, pts * 3 * sizeof(float), cudaMemcpyDeviceToHost, cp));
    HG_CUDA(cudaMemcpyAsync(s->loss_pinned + b0, sl.total, (size_t)nb * sizeof(float), cudaMemcpyDeviceToHost, cp));
  }
  HG_CUDA(cudaStreamSynchronize(s->slot[0].stream));
  HG_CUDA(cudaStreamSynchronize(s->slot[1].stream));
  HG_CUDA(cudaStreamSynchronize(s->compute));
  double acc = 0.0;
  for (int b = 0; b < B; ++b) {
    cloud_loss_h[b] = s->loss_pinned[b];
    acc += (double)cloud_loss_h[b];
  }
  *loss_h = (float)(acc / (double)B);
  return HG_OK;
}
