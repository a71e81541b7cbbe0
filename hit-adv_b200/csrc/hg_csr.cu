// hg_csr.cu -- deterministic reverse map for scatter-style backward passes.
//
// The reference accumulates every scatter gradient with float atomicAdd (sampling_gpu.cu:43,
// group_points_gpu.cu:60, interpolate_gpu.cu:139-141) or with ATen index_put(accumulate=True); the sum
// order, and therefore the low bits of the result, change from run to run.  Here each destination gets the
// list of its source edges in ascending edge order (a stable counting sort per cloud); consumers add in
// list order, so results are bit-reproducible.  Integer atomics (counts) are order-independent.
#include "hg_common.cuh"

namespace {

constexpr int kCsrThreads = 256;
constexpr int kCsrWarps = kCsrThreads / 32;

// One CTA per cloud.  The edge range is cut into kCsrWarps contiguous segments, one per warp: per-warp key
// counts -> exclusive prefix over (key, warp) -> every warp places its own segment stably (chunks of 32 edges in
// ascending order, rank inside a chunk from __match_any_sync), all warps in parallel.
__global__ void __launch_bounds__(kCsrThreads) csr_build_kernel(const int *__restrict__ keys, int E, int N,
                                                                int *__restrict__ off_all,
                                                                int *__restrict__ cursor_all,
                                                                int *__restrict__ list_all) {
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nbits = 32 - __clz(N);  // keys 0..N (N = invalid) fit
  const int *k = keys + (size_t)b * E;
  int *off = off_all + (size_t)b * (N + 1);
  int *cursor = cursor_all + (size_t)b * kCsrWarps * N;  // [kCsrWarps][N]
  int *list = list_all + (size_t)b * E;
  __shared__ int warp_tot[kCsrWarps];
  __shared__ int carry_s;

  const int seg = ((E + kCsrWarps - 1) / kCsrWarps + 31) / 32 * 32;  // edges per warp segment (multiple of 32)
  const int e_lo = min(E, warp * seg), e_hi = min(E, (warp + 1) * seg);
  int *mine = cursor + (size_t)warp * N;

  for (int i = tid; i <= N; i += kCsrThreads) off[i] = 0;
  for (int i = tid; i < kCsrWarps * N; i += kCsrThreads) cursor[i] = 0;
  __syncthreads();
  for (int e = e_lo + lane; e < e_hi; e += 32) {
    const int key = k[e];
    if (key >= 0 && key < N) {
      atomicAdd(&off[key + 1], 1);
      atomicAdd(&mine[key], 1);
    }
  }
  if (tid == 0) carry_s = 0;
  __syncthreads();
  // inclusive scan of off[1..N] (off[0] stays 0) -> off[i] = #edges with key < i
  for (int base = 1; base <= N; base += kCsrThreads) {
    const int i = base + tid;
    int v = (i <= N) ? off[i] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int add = carry_s;
    for (int w = 0; w < warp; ++w) add += warp_tot[w];
    if (i <= N) off[i] = v + add;
    __syncthreads();
    if (tid == kCsrThreads - 1) carry_s = v + add;
    __syncthreads();
  }
  // per-warp start of every key: segment start + edges of that key in the earlier warps' segments
  for (int key = tid; key < N; key += kCsrThreads) {
    int run = off[key];
    for (int w = 0; w < kCsrWarps; ++w) {
      const int c = cursor[(size_t)w * N + key];
      cursor[(size_t)w * N + key] = run;
      run += c;
    }
  }
  __syncthreads();
  for (int base = e_lo; base < e_hi; base += 32) {
    const int e = base + lane;
    int key = (e < e_hi) ? k[e] : -1;
    if (key >= N || key < 0) key = N;  // N = "no key": fits the nbits of the ballot match
    const unsigned same = hg_match_any_bits(key, nbits);
    const int rank = __popc(same & ((1u << lane) - 1u));
    int pos = 0;
    if (key < N) pos = mine[key] + rank;
    __syncwarp();
    if (key < N) {
      list[pos] = e;
      if (rank == 0) mine[key] = pos + __popc(same);
    }
    __syncwarp();
  }
}

// ---- the same build with the per-warp cursors in shared memory -----------------------------------------------------
// In the kernel above every placement step is a dependent round trip through global memory (read the segment's cursor
// for the key, store the edge, write the cursor back): 64 such steps per warp at 16k edges per cloud, ~70 us whatever
// the batch.  With the kCsrWarps x N cursors (and the key counts) in shared memory the same steps cost a shared-memory
// latency each, and the CTA can afford MORE segments (W = 8, 16 or 32 warps: the chain of dependent steps per warp
// shrinks accordingly; the stable order does not depend on how the edge range is cut).  Same list, bit for bit.  Needs
// (W + 1) * N + 1 ints of shared memory, plus E ints when the keys are staged as well.
template <int W>
__global__ void __launch_bounds__(32 * W) csr_build_smem_kernel(const int *__restrict__ keys, int E, int N,
                                                                     int *__restrict__ off_all,
                                                                     int *__restrict__ list_all, int stage_keys) {
  extern __shared__ int csm[];
  int *soff = csm;                 // [N+1]
  int *cursor = csm + (N + 1);     // [W][N]
  int *skeys = csm + (((size_t)(W + 1) * N + 1 + 3) & ~(size_t)3);  // [E], 16-byte aligned, when stage_keys: the count and placement loops below are
                                                // latency-bound, one dependent step per 32 edges -- with the keys
                                                // read from global memory every step pays a DRAM/L2 round trip
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nbits = 32 - __clz(N);  // keys 0..N (N = invalid) fit
  const int *k = keys + (size_t)b * E;
  if (stage_keys) {
    if ((E & 3) == 0 && (reinterpret_cast<uintptr_t>(k) & 15) == 0) {  // 16 bytes per load, four loads in flight
      const int4 *k4 = reinterpret_cast<const int4 *>(k);
      int4 *s4 = reinterpret_cast<int4 *>(skeys);
      int e = tid;
      for (; e + 3 * (32 * W) < E / 4; e += 4 * (32 * W)) {
        const int4 a = k4[e], b4 = k4[e + (32 * W)], c4 = k4[e + 2 * (32 * W)], d4 = k4[e + 3 * (32 * W)];
        s4[e] = a;
        s4[e + (32 * W)] = b4;
        s4[e + 2 * (32 * W)] = c4;
        s4[e + 3 * (32 * W)] = d4;
      }
      for (; e < E / 4; e += (32 * W)) s4[e] = k4[e];
    } else {
      for (int e = tid; e < E; e += (32 * W)) skeys[e] = k[e];
    }
    k = skeys;
  }
  int *off = off_all + (size_t)b * (N + 1);
  int *list = list_all + (size_t)b * E;
  __shared__ int warp_tot[W];
  __shared__ int carry_s;

  const int seg = ((E + W - 1) / W + 31) / 32 * 32;  // edges per warp segment (multiple of 32)
  const int e_lo = min(E, warp * seg), e_hi = min(E, (warp + 1) * seg);
  int *mine = cursor + (size_t)warp * N;

  for (int i = tid; i < (W + 1) * N + 1; i += (32 * W)) csm[i] = 0;
  __syncthreads();
  // per-segment key counts WITHOUT atomics (a shared-memory atomic costs ~2 cycles per lane, and there would be two per
  // edge): the segment's counters belong to this warp alone, so the lanes of a step that share a key elect a leader
  // (match_any) which does a plain read-modify-write
  for (int base = e_lo; base < e_hi; base += 32) {
    const int e = base + lane;
    int key = (e < e_hi) ? k[e] : -1;
    if (key >= N || key < 0) key = N;
    const unsigned same = hg_match_any_bits(key, nbits);
    if (key < N && (same & ((1u << lane) - 1u)) == 0u) mine[key] += __popc(same);
    __syncwarp();
  }
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int key = tid; key < N; key += (32 * W)) {  // key totals over the segments
    int t = 0;
#pragma unroll
    for (int w = 0; w < W; ++w) t += cursor[(size_t)w * N + key];
    soff[key + 1] = t;
  }
  __syncthreads();
  for (int base = 1; base <= N; base += (32 * W)) {  // inclusive scan of soff[1..N] -> soff[i] = #edges with key < i
    const int i = base + tid;
    int v = (i <= N) ? soff[i] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int add = carry_s;
    for (int w = 0; w < warp; ++w) add += warp_tot[w];
    if (i <= N) soff[i] = v + add;
    __syncthreads();
    if (tid == (32 * W) - 1) carry_s = v + add;
    __syncthreads();
  }
  for (int i = tid; i <= N; i += (32 * W)) off[i] = soff[i];
  for (int key = tid; key < N; key += (32 * W)) {  // start of every (warp segment, key) run
    int run = soff[key];
#pragma unroll
    for (int w = 0; w < W; ++w) {
      const int c = cursor[(size_t)w * N + key];
      cursor[(size_t)w * N + key] = run;
      run += c;
    }
  }
  __syncthreads();
  for (int base = e_lo; base < e_hi; base += 32) {
    const int e = base + lane;
    int key = (e < e_hi) ? k[e] : -1;
    if (key >= N || key < 0) key = N;  // N = "no key": fits the nbits of the ballot match
    const unsigned same = hg_match_any_bits(key, nbits);
    const int rank = __popc(same & ((1u << lane) - 1u));
    int pos = 0;
    if (key < N) pos = mine[key] + rank;
    __syncwarp();
    if (key < N) {
      list[pos] = e;
      if (rank == 0) mine[key] = pos + __popc(same);
    }
    __syncwarp();
  }
}

}  // namespace

// Tiny problems (a couple of thousand edges per cloud) are launch-bound: one stable single-kernel build beats memset +
// count + scan + fill.  Beyond that the single CTA per cloud of the stable builder is the bottleneck (48 us against
// ~20 us for 388 clouds x 6144 edges).  hg_csr_build_unordered switches on this and the workspace formula follows it.
static inline bool csr_small(int E) { return E <= 2048; }

// off [B,N+1], cursors (kCsrWarps per key for the stable builder, one for the atomic one), list [B,E]
struct CsrLayout {
  int *off, *cursor, *list;
  CsrLayout(HgCarve &c, int B, int N, int E, bool stable)
      : off(c.take<int>((size_t)B * (N + 1))), cursor(c.take<int>((size_t)B * (stable ? kCsrWarps : 1) * N)),
        list(c.take<int>((size_t)B * E)) {}
};

size_t hg_csr_workspace_bytes(int B, int N, int E) {
  return hg_layout_bytes<CsrLayout>(B, N, E, csr_small(E));
}

size_t hg_csr_stable_workspace_bytes(int B, int N, int E) {
  return hg_layout_bytes<CsrLayout>(B, N, E, true);
}

int hg_csr_build(const int *keys, int B, int E, int N, void *workspace, size_t workspace_bytes, HgCsr *out,
                 cudaStream_t stream) {
  HG_REQUIRE(workspace && workspace_bytes >= hg_csr_stable_workspace_bytes(B, N, E), HG_E_WORKSPACE,
             "csr: workspace too small (%zu < %zu)", workspace_bytes, hg_csr_stable_workspace_bytes(B, N, E));
  const auto [off, cursor, list] = hg_layout_at<CsrLayout>(workspace, B, N, E, true);
  {
    // most warps whose cursors (and, if possible, the staged keys) fit in shared memory
    auto need = [&](int w, bool keys_too) {
      return (((size_t)(w + 1) * N + 1 + 3) & ~(size_t)3) * sizeof(int) + (keys_too ? (size_t)E * sizeof(int) : 0);
    };
    const size_t limit = 200 * 1024;
    int W = 0, stage_keys = 0;
    const int want = E >= 8192 ? 32 : (E >= 2048 ? 16 : 8);
    for (int w = want; w >= 8 && !W; w >>= 1)
      if (need(w, true) <= limit) W = w, stage_keys = 1;
    for (int w = want; w >= 8 && !W; w >>= 1)
      if (need(w, false) <= limit) W = w;
    if (W) {
      const size_t smem = need(W, stage_keys != 0);
      static HgPerDeviceOnce once;
      if (once.first()) {
        HG_CUDA(cudaFuncSetAttribute(csr_build_smem_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
        HG_CUDA(cudaFuncSetAttribute(csr_build_smem_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
        HG_CUDA(cudaFuncSetAttribute(csr_build_smem_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)limit));
      }
      if (W == 32)
        csr_build_smem_kernel<32><<<B, 1024, smem, stream>>>(keys, E, N, off, list, stage_keys);
      else if (W == 16)
        csr_build_smem_kernel<16><<<B, 512, smem, stream>>>(keys, E, N, off, list, stage_keys);
      else
        csr_build_smem_kernel<8><<<B, 256, smem, stream>>>(keys, E, N, off, list, stage_keys);
      HG_CHECK_LAUNCH("csr_build_smem_kernel");
      out->off = off;
      out->list = list;
      return HG_OK;
    }
  }
  csr_build_kernel<<<B, kCsrThreads, 0, stream>>>(keys, E, N, off, cursor, list);
  HG_CHECK_LAUNCH("csr_build_kernel");
  out->off = off;
  out->list = list;
  return HG_OK;
}

// ---- unordered variant for the hot-loop backward passes ---------------------------------------------------------
// Same off/list layout, but the position of an edge inside its destination's segment is taken from an integer
// atomic (fully parallel over the edges, no serial placement).  Consumers then walk a segment in ascending edge
// order with hg_csr_next() (selection over the few entries), so the summation order -- and the result -- is still
// independent of how the atomics resolved.  Segments are tiny on this path (Chamfer: multiplicity <= ~3; kNN:
// only edges leaving outlier points), which is what makes the O(c^2) walk cheaper than a stable sort.
namespace {

__global__ void __launch_bounds__(256) csr_count_kernel(const int *__restrict__ keys, long long total, int E, int N,
                                                        int *__restrict__ off_all) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int key = keys[g];
    if (key >= 0 && key < N) atomicAdd(off_all + (g / E) * (N + 1) + key + 1, 1);
  }
}

__global__ void __launch_bounds__(256) csr_scan_kernel(int N, int *__restrict__ off_all, int *__restrict__ cursor_all) {
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int *off = off_all + (size_t)b * (N + 1);
  int *cursor = cursor_all + (size_t)b * N;
  __shared__ int warp_tot[8];
  __shared__ int carry_s;
  if (tid == 0) carry_s = 0;
  __syncthreads();
  for (int base = 1; base <= N; base += 256) {
    const int i = base + tid;
    int v = (i <= N) ? off[i] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int add = carry_s;
    for (int w = 0; w < warp; ++w) add += warp_tot[w];
    if (i <= N) {
      off[i] = v + add;
      if (i < N) cursor[i] = v + add;  // start of segment i
    }
    __syncthreads();
    if (tid == 255) carry_s = v + add;
    __syncthreads();
  }
  if (tid == 0) cursor[0] = 0;
}

__global__ void __launch_bounds__(256) csr_fill_kernel(const int *__restrict__ keys, long long total, int E, int N,
                                                       int *__restrict__ cursor_all, int *__restrict__ list_all) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int key = keys[g];
    if (key >= 0 && key < N) {
      const long long b = g / E;
      const int pos = atomicAdd(cursor_all + b * N + key, 1);
      list_all[b * E + pos] = (int)(g - b * E);
    }
  }
}

}  // namespace

int hg_csr_build_unordered(const int *keys, int B, int E, int N, void *workspace, size_t workspace_bytes, HgCsr *out,
                           cudaStream_t stream) {
  HG_REQUIRE(workspace && workspace_bytes >= hg_csr_workspace_bytes(B, N, E), HG_E_WORKSPACE,
             "csr: workspace too small (%zu < %zu)", workspace_bytes, hg_csr_workspace_bytes(B, N, E));
  if (csr_small(E)) return hg_csr_build(keys, B, E, N, workspace, workspace_bytes, out, stream);  // sorted is fine too
  const auto [off, cursor, list] = hg_layout_at<CsrLayout>(workspace, B, N, E, false);
  HG_CUDA(cudaMemsetAsync(off, 0, (size_t)B * (N + 1) * sizeof(int), stream));
  const long long total = (long long)B * E;
  const int blocks = hg_grid_for(total, 256, 16);
  csr_count_kernel<<<blocks, 256, 0, stream>>>(keys, total, E, N, off);
  HG_CHECK_LAUNCH("csr_count_kernel");
  csr_scan_kernel<<<B, 256, 0, stream>>>(N, off, cursor);
  HG_CHECK_LAUNCH("csr_scan_kernel");
  csr_fill_kernel<<<blocks, 256, 0, stream>>>(keys, total, E, N, cursor, list);
  HG_CHECK_LAUNCH("csr_fill_kernel");
  out->off = off;
  out->list = list;
  return HG_OK;
}
