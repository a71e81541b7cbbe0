// hg_pointnet2.cu -- the nine pointnet2_ops kernels (pointnet2_ops_lib/pointnet2_ops/_ext-src/src/*.cu),
// rewritten for sm_100a behind the reference's own C-style wrapper signatures, and the torch-level FPS of
// model/pointnet2_utils.py:63-84 (same kernel, different arithmetic / tie rule).
//
// What changes w.r.t. the reference kernels (which launch ONE CTA per batch element, <= b of 148 SMs busy):
//   * gather / group / interpolate: one thread per output element over the whole grid, coalesced stores;
//   * *_grad: deterministic segmented sums over a reverse map (hg_csr.cu) instead of float atomicAdd;
//   * ball query: a warp per centre scanning 32 points per step (ballot + prefix popcount keep the
//     ascending-index order of the serial reference loop), early exit once nsample hits are found;
//   * FPS: the cloud and the running distances live in registers for the whole launch, one 64-bit
//     (distance, tie-key) max per round, ONE barrier per round (double-buffered warp results) instead of the
//     reference's 10; the tie key reproduces the reference's shared-memory tree order exactly.
// Index results are bit-identical to the reference kernels (same FMA contraction as nvcc emits for them).
#include "hg_common.cuh"

namespace {

// cuda_utils.h:13-17 opt_n_threads -- only its value matters here: it fixes the reference FPS tie order.
int ref_opt_n_threads(int work_size) {
  const int pow_2 = (int)(std::log((double)work_size) / std::log(2.0));
  int t = 1 << pow_2;
  if (t > 512) t = 512;
  if (t < 1) t = 1;
  return t;
}

// ---- gather / group (sampling_gpu.cu:8-20, group_points_gpu.cu:8-28) ---------------------------------------
// out[b,c,e] = points[b,c,idx[b,e]],  e over the flattened index tensor (m, or npoints*nsample).
// HBM-bound on the output write: four consecutive e per thread (one int4 index load, four gathers per channel, one
// streaming float4 store per channel), no integer division.
// SMEM: the source planes (n floats each) are staged in shared memory first -- random 4-byte gathers from L1 cost one
// wavefront per distinct line and cap the kernel near 2 TB/s; from shared memory they cost a few bank cycles.
// A CTA pass covers kGatherCP channels of one cloud, so that every index load serves kGatherCP output rows.
constexpr int kGatherCP = 4;
template <bool VEC4, bool SMEM>
__global__ void __launch_bounds__(256) gather_channel_major_kernel(const float *__restrict__ points,
                                                                   const int *__restrict__ idx, int c, int n, int E,
                                                                   long long groups, float *__restrict__ out,
                                                                   int oc_total, int oc_off) {
  extern __shared__ float plane[];  // SMEM: [kGatherCP][n]
  const int gpc = (c + kGatherCP - 1) / kGatherCP;  // channel groups per cloud
  for (long long gi = blockIdx.y; gi < groups; gi += gridDim.y) {
    const long long bi = gi / gpc;
    const int c0 = (int)(gi % gpc) * kGatherCP;
    const int nc = min(kGatherCP, c - c0);
    const float *src = points + ((size_t)bi * c + c0) * n;
    const int *id = idx + (size_t)bi * E;
    float *dst = out + ((size_t)bi * oc_total + oc_off + c0) * E;  // (oc_total, oc_off): a channel slice of a wider output
    if (SMEM) {
      __syncthreads();
      for (int k = threadIdx.x; k < nc * n; k += 256) plane[k] = __ldg(src + k);
      __syncthreads();
    }
    const float *tab = SMEM ? plane : src;
    if (VEC4) {
      const int step = gridDim.x * 1024;
      int e = (blockIdx.x * 256 + threadIdx.x) * 4;
      for (; e + step < E; e += 2 * step) {  // two index loads in flight per thread
        const int4 a0 = *reinterpret_cast<const int4 *>(id + e), a1 = *reinterpret_cast<const int4 *>(id + e + step);
#pragma unroll
        for (int q = 0; q < kGatherCP; ++q)
          if (q < nc) {
            const float *t = tab + (size_t)q * n;
            __stcs(reinterpret_cast<float4 *>(dst + (size_t)q * E + e), make_float4(t[a0.x], t[a0.y], t[a0.z], t[a0.w]));
            __stcs(reinterpret_cast<float4 *>(dst + (size_t)q * E + e + step),
                   make_float4(t[a1.x], t[a1.y], t[a1.z], t[a1.w]));
          }
      }
      for (; e < E; e += step) {
        const int4 a = *reinterpret_cast<const int4 *>(id + e);
#pragma unroll
        for (int q = 0; q < kGatherCP; ++q)
          if (q < nc) {
            const float *t = tab + (size_t)q * n;
            __stcs(reinterpret_cast<float4 *>(dst + (size_t)q * E + e), make_float4(t[a.x], t[a.y], t[a.z], t[a.w]));
          }
      }
    } else {
      for (int e = blockIdx.x * 256 + threadIdx.x; e < E; e += gridDim.x * 256) {
        const int a = __ldg(id + e);
        for (int q = 0; q < nc; ++q) dst[(size_t)q * E + e] = tab[(size_t)q * n + a];
      }
    }
  }
}

int launch_gather(const float *points, const int *idx, int b, int c, int n, int E, float *out, cudaStream_t stream,
                  int prof_tag, int oc_total = 0, int oc_off = 0) {
  if (oc_total == 0) oc_total = c;
  const long long groups = (long long)b * ((c + kGatherCP - 1) / kGatherCP);
  const bool vec = (E % 4 == 0) && ((reinterpret_cast<uintptr_t>(idx) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  const int per_block = vec ? 1024 : 256;
  // stage the planes when they are re-used enough (E >= n) and fit
  const bool use_smem = (size_t)kGatherCP * n * sizeof(float) <= 96 * 1024 && E >= n;
  int gx = (E + per_block - 1) / per_block;
  // enough CTAs to fill the machine a few times over; with staged planes each CTA amortises its staging over >= 1/gx
  // of the indices
  long long gx_cap = use_smem ? (8LL * hg_sm_count() + groups - 1) / groups : 64;
  if (gx_cap < 1) gx_cap = 1;
  if (gx > gx_cap) gx = (int)gx_cap;
  const int gy = (int)(groups < 65535 ? groups : 65535);
  const size_t smem = use_smem ? (size_t)kGatherCP * n * sizeof(float) : 0;
  const bool prof = prof_tag >= 0 ? hg_prof_begin(prof_tag, stream) : false;
#define HG_GATHER_LAUNCH(V, S)                                                                                     \
  do {                                                                                                             \
    if (smem > 48 * 1024)                                                                                          \
      cudaFuncSetAttribute(gather_channel_major_kernel<V, S>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
    gather_channel_major_kernel<V, S><<<dim3(gx, gy), 256, smem, stream>>>(points, idx, c, n, E, groups, out,      \
                                                                           oc_total, oc_off);                      \
  } while (0)
  if (vec && use_smem) HG_GATHER_LAUNCH(true, true);
  else if (vec) HG_GATHER_LAUNCH(true, false);
  else if (use_smem) HG_GATHER_LAUNCH(false, true);
  else HG_GATHER_LAUNCH(false, false);
#undef HG_GATHER_LAUNCH
  hg_prof_end(prof_tag, stream, prof);
  HG_CHECK_LAUNCH("gather_channel_major_kernel");
  return HG_OK;
}

// grad_points[b,c,key] = sum over the edges e of key, ascending e, of src[b,c,e / DIV] * (w ? w[b,e] : 1)
template <int DIV, bool WEIGHTED>
__global__ void __launch_bounds__(256) scatter_channel_major_kernel(const float *__restrict__ src,
                                                                    const float *__restrict__ w,
                                                                    const int *__restrict__ off,
                                                                    const int *__restrict__ list, int b, int c, int n,
                                                                    int E, float *__restrict__ grad_points,
                                                                    int sc_total = 0, int sc_off = 0) {
  const long long total = (long long)b * c * n;
  const int Esrc = E / DIV;
  if (sc_total == 0) sc_total = c;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int key = (int)(g % n);
    const long long bc = g / n;
    const int bi = (int)(bc / c);
    const int *o = off + (size_t)bi * (n + 1);
    const int *l = list + (size_t)bi * E;
    const float *s = src + ((size_t)bi * sc_total + sc_off + (int)(bc % c)) * Esrc;
    float acc = 0.f;
    for (int q = o[key]; q < o[key + 1]; ++q) {
      const int e = l[q];
      float v = s[e / DIV];
      if (WEIGHTED) v = __fmul_rn(v, w[(size_t)bi * E + e]);
      acc = __fadd_rn(acc, v);
    }
    grad_points[g] = acc;
  }
}

// Staged variant for the gather / group gradients (DIV = 1, unweighted): one CTA per (b,c) plane copies the plane's E
// source values into shared memory with coalesced float4 loads, then every thread sums its destination's incoming
// edges from shared memory (the generic kernel above gathers 4 bytes per 32-byte sector from global memory).  Same
// sequential summation order (ascending edge) => the same bits as the generic kernel and the oracle.
constexpr int kScatterThreads = 256;
__global__ void __launch_bounds__(kScatterThreads) scatter_staged_kernel(const float *__restrict__ src,
                                                                         const int *__restrict__ off,
                                                                         const int *__restrict__ list, int c, int n, int E,
                                                                         long long planes, float *__restrict__ grad_points,
                                                                         int sc_total, int sc_off) {
  extern __shared__ float sA[];  // [E]
  for (long long bc = blockIdx.x; bc < planes; bc += gridDim.x) {
    const long long bi = bc / c;
    const float *s = src + ((size_t)bi * sc_total + sc_off + (int)(bc % c)) * E;  // a channel slice of a wider source
    const int *o = off + (size_t)bi * (n + 1);
    const int *l = list + (size_t)bi * E;
    float *dst = grad_points + (size_t)bc * n;
    __syncthreads();
    if ((E & 3) == 0 && (reinterpret_cast<uintptr_t>(s) & 15) == 0) {
      for (int e = threadIdx.x * 4; e < E; e += kScatterThreads * 4)
        *reinterpret_cast<float4 *>(sA + e) = __ldcs(reinterpret_cast<const float4 *>(s + e));
    } else {
      for (int e = threadIdx.x; e < E; e += kScatterThreads) sA[e] = s[e];
    }
    __syncthreads();
    for (int key = threadIdx.x; key < n; key += kScatterThreads) {
      const int q1 = o[key + 1];
      int q = o[key];
      float acc = 0.f;
      for (; q + 3 < q1; q += 4) {  // four list entries in flight
        const int e0 = __ldg(l + q), e1 = __ldg(l + q + 1), e2 = __ldg(l + q + 2), e3 = __ldg(l + q + 3);
        acc = __fadd_rn(acc, sA[e0]);
        acc = __fadd_rn(acc, sA[e1]);
        acc = __fadd_rn(acc, sA[e2]);
        acc = __fadd_rn(acc, sA[e3]);
      }
      for (; q < q1; ++q) acc = __fadd_rn(acc, sA[__ldg(l + q)]);
      dst[key] = acc;
    }
  }
}

// The same sums with the planes streamed by the copy engine: a CTA owns a contiguous run of (b,c) planes (the reverse
// map of a cloud stays in L1 across its channels) and double-buffers them in shared memory -- while the 256 threads sum
// plane i out of one buffer, ONE cp.async.bulk (UBLKCP) brings the whole of plane i+1 into the other, completion on an
// mbarrier.  The staged kernel above loads, barriers, computes, barriers: its loads never overlap its sums.
constexpr int kBulkThreads = 1024, kBulkWarps = kBulkThreads / 32;
// LIST_SMEM: the reverse map of the current cloud (shared by its c planes) also lives in shared memory, re-laid-out so
// that a warp reads it without bank conflicts: the lists of 32 consecutive keys are interleaved ("sliced ELL":
// entry j of key 32*blk + lane sits at base[blk] + 32*j + lane, each block padded to its longest list), 16 bits per
// entry.  Read from global memory every batch of entries is an L2 round trip in the middle of a dependent chain; kept
// in CSR order in shared memory, lanes whose lists start ~deg entries apart collide on a handful of banks (ncu: 57 %
// of the kernel's shared-memory wavefronts were conflict replays).  A cloud whose padded lists do not fit (hub keys)
// falls back to the global-memory walk for that cloud.
template <bool LIST_SMEM>
__global__ void __launch_bounds__(kBulkThreads) scatter_bulk_kernel(const float *__restrict__ src,
                                                                    const int *__restrict__ off,
                                                                    const int *__restrict__ list, int c, int n, int E,
                                                                    long long planes, float *__restrict__ grad_points,
                                                                    int sc_total, int sc_off, int cap /*ELL entries*/) {
  extern __shared__ __align__(128) float sB[];  // [2][E] planes, then (LIST_SMEM) so [n+1], sbase [nblk+1], ELL [cap]
  const int nblk = (n + 31) / 32;
  int *so = reinterpret_cast<int *>(sB + 2 * (size_t)E);
  int *sbase = so + (n + 1);
  unsigned short *sl = reinterpret_cast<unsigned short *>(sbase + (nblk + 1));
  __shared__ __align__(8) uint64_t bar[2];
  __shared__ int ell_ok;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long per = (planes + gridDim.x - 1) / gridDim.x;
  const long long p_lo = (long long)blockIdx.x * per, p_hi = min(planes, p_lo + per);
  if (p_lo >= p_hi) return;
  const unsigned bytes = (unsigned)E * sizeof(float);
  auto plane_src = [&](long long bc) { return src + ((size_t)(bc / c) * sc_total + sc_off + (int)(bc % c)) * E; };
  if (threadIdx.x == 0) {
    hg_mbar_init(&bar[0], 1);
    hg_mbar_init(&bar[1], 1);
    hg_mbar_init_fence();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    hg_mbar_expect_tx(&bar[0], bytes);
    hg_bulk_g2s(sB, plane_src(p_lo), bytes, &bar[0]);
  }
  int it = 0;
  long long cloud = -1;
  for (long long bc = p_lo; bc < p_hi; ++bc, ++it) {
    const int cur = it & 1;
    if (threadIdx.x == 0 && bc + 1 < p_hi) {  // the other buffer was released by the barrier that ended iteration it-1
      hg_mbar_expect_tx(&bar[cur ^ 1], bytes);
      hg_bulk_g2s(sB + (size_t)(cur ^ 1) * E, plane_src(bc + 1), bytes, &bar[cur ^ 1]);
    }
    const long long bi = bc / c;
    const int *o = off + (size_t)bi * (n + 1);
    const int *l = list + (size_t)bi * E;
    if (LIST_SMEM && bi != cloud) {  // new cloud: build its interleaved map
      cloud = bi;
      for (int i = threadIdx.x; i <= n; i += kBulkThreads) so[i] = o[i];
      __syncthreads();
      for (int blk = warp; blk < nblk; blk += kBulkWarps) {  // longest list of every block of 32 keys
        const int key = blk * 32 + lane;
        const int deg = key < n ? so[key + 1] - so[key] : 0;
        const int m = __reduce_max_sync(0xffffffffu, deg);
        if (lane == 0) sbase[blk + 1] = 32 * m;
      }
      __syncthreads();
      if (warp == 0) {  // exclusive prefix over the blocks
        int run = 0;
        for (int b0 = 0; b0 < nblk; b0 += 32) {
          const int i = b0 + lane;
          const int v = i < nblk ? sbase[i + 1] : 0;
          int incl = v;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
          }
          if (i < nblk) sbase[i + 1] = run + incl;
          run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) {
          sbase[0] = 0;
          ell_ok = run <= cap;
        }
      }
      __syncthreads();
      if (ell_ok) {
        for (int blk = warp; blk < nblk; blk += kBulkWarps) {
          const int key = blk * 32 + lane;
          const int q0 = key < n ? so[key] : 0, deg = key < n ? so[key + 1] - q0 : 0;
          unsigned short *dst = sl + sbase[blk] + lane;
          for (int j = 0; j < deg; ++j) dst[32 * j] = (unsigned short)__ldg(l + q0 + j);
        }
      }
      __syncthreads();
    }
    hg_mbar_wait(&bar[cur], (unsigned)(it >> 1) & 1u);
    const float *sA = sB + (size_t)cur * E;
    float *dst = grad_points + (size_t)bc * n;
    if (LIST_SMEM && ell_ok) {
      for (int blk = warp; blk < nblk; blk += kBulkWarps) {
        const int key = blk * 32 + lane;
        const int deg = key < n ? so[key + 1] - so[key] : 0;
        const unsigned short *lp = sl + sbase[blk] + lane;
        float acc = 0.f;
        int j = 0;
        for (; j + 3 < deg; j += 4) {  // four entries in flight; the sum itself stays sequential (ascending edge)
          const int e0 = lp[32 * j], e1 = lp[32 * j + 32], e2 = lp[32 * j + 64], e3 = lp[32 * j + 96];
          const float v0 = sA[e0], v1 = sA[e1], v2 = sA[e2], v3 = sA[e3];
          acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v0), v1), v2), v3);
        }
        for (; j < deg; ++j) acc = __fadd_rn(acc, sA[lp[32 * j]]);
        if (key < n) dst[key] = acc;
      }
    } else {
      for (int key = threadIdx.x; key < n; key += kBulkThreads) {
        const int q1 = o[key + 1];
        int q = o[key];
        float acc = 0.f;
        for (; q + 3 < q1; q += 4) {
          const int e0 = __ldg(l + q), e1 = __ldg(l + q + 1), e2 = __ldg(l + q + 2), e3 = __ldg(l + q + 3);
          const float v0 = sA[e0], v1 = sA[e1], v2 = sA[e2], v3 = sA[e3];
          acc = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(acc, v0), v1), v2), v3);
        }
        for (; q < q1; ++q) acc = __fadd_rn(acc, sA[__ldg(l + q)]);
        dst[key] = acc;
      }
    }
    __syncthreads();  // every thread is done with this buffer (and this cloud's map) before the copy engine refills it
  }
}

// gradient of gather / group: bulk-copy pipeline when two planes fit in shared memory (and the planes are 16-byte
// aligned), single-buffer staged kernel when one does, generic kernel otherwise
int launch_scatter_unweighted(const float *grad_out, const HgCsr &csr, int b, int c, int n, int E, float *grad_points,
                              cudaStream_t stream, int sc_total = 0, int sc_off = 0) {
  if (sc_total == 0) sc_total = c;
  const size_t smem = (size_t)E * sizeof(float);
  const long long planes = (long long)b * c;
  const bool bulk_ok = 2 * smem <= 200 * 1024 && E >= n && (E & 3) == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 15) == 0;
  if (bulk_ok && planes >= 2LL * hg_sm_count()) {
    static HgPerDeviceOnce once;
    if (once.first()) {
      HG_CUDA(cudaFuncSetAttribute(scatter_bulk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
      HG_CUDA(cudaFuncSetAttribute(scatter_bulk_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    }
    // shared memory beyond the two plane buffers goes to the cloud's interleaved map: it needs ~1.6 E entries for
    // Poisson-like in-degrees (longest of 32 lists); take what is there, the kernel falls back per cloud if it overflows
    const size_t fixed = 2 * smem + ((size_t)(n + 1) + (size_t)((n + 31) / 32 + 1)) * sizeof(int);
    const size_t limit = 220 * 1024;
    long long cap = fixed < limit ? (long long)((limit - fixed) / sizeof(unsigned short)) : 0;
    if (cap > 4LL * E) cap = 4LL * E;
    const bool list_smem = cap >= (long long)E + 32LL * ((n + 31) / 32) && E <= 65535;
    const size_t dyn = list_smem ? fixed + (size_t)cap * sizeof(unsigned short) : 2 * smem;
    const int per_sm = (dyn <= 100 * 1024) ? 2 : 1;
    long long grid = (long long)hg_sm_count() * per_sm;
    if (grid > planes) grid = planes;
    if (list_smem)
      scatter_bulk_kernel<true><<<(int)grid, kBulkThreads, dyn, stream>>>(grad_out, csr.off, csr.list, c, n, E, planes,
                                                                         grad_points, sc_total, sc_off, (int)cap);
    else
      scatter_bulk_kernel<false><<<(int)grid, kBulkThreads, dyn, stream>>>(grad_out, csr.off, csr.list, c, n, E, planes,
                                                                          grad_points, sc_total, sc_off, 0);
  } else if (smem <= 100 * 1024 && E >= n) {  // (two CTAs per SM)
    if (smem > 48 * 1024)
      HG_CUDA(cudaFuncSetAttribute(scatter_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long grid = planes;
    const long long cap = (long long)hg_sm_count() * 8;
    if (grid > cap) grid = cap;
    scatter_staged_kernel<<<(int)grid, kScatterThreads, smem, stream>>>(grad_out, csr.off, csr.list, c, n, E, planes,
                                                                       grad_points, sc_total, sc_off);
  } else {
    const long long total = (long long)b * c * n;
    scatter_channel_major_kernel<1, false><<<hg_grid_for(total, 256, 32), 256, 0, stream>>>(grad_out, nullptr, csr.off, csr.list,
                                                                                            b, c, n, E, grad_points, sc_total,
                                                                                            sc_off);
  }
  return HG_OK;
}

// QueryAndGroup's coordinate rows: out[b, d, s, t] = xyz[b, idx[b,s,t], d] - new_xyz[b, s, d], d < 3, written into the
// first three channels of the (b, oc_total, S, ns) output
__global__ void __launch_bounds__(256) group_xyz_rel_kernel(const float *__restrict__ xyz,
                                                            const float *__restrict__ new_xyz,
                                                            const int *__restrict__ idx, int n, int S, int ns,
                                                            int oc_total, long long total, float *__restrict__ out) {
  const int E = S * ns;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long bi = g / E;
    const int e = (int)(g % E), sidx = e / ns;
    const int a = __ldg(idx + g);
    const float *p = xyz + ((size_t)bi * n + a) * 3;
    const float *q = new_xyz + ((size_t)bi * S + sidx) * 3;
    float *o = out + (size_t)bi * oc_total * E + e;
    o[0] = __fsub_rn(__ldg(p), __ldg(q));
    o[(size_t)E] = __fsub_rn(__ldg(p + 1), __ldg(q + 1));
    o[(size_t)2 * E] = __fsub_rn(__ldg(p + 2), __ldg(q + 2));
  }
}

// ---- ball query (ball_query_gpu.cu:9-44) -------------------------------------------------------------------
__global__ void __launch_bounds__(128) ball_query_kernel(int n, int m, float radius2, int nsample,
                                                         const float *__restrict__ new_xyz,
                                                         const float *__restrict__ xyz, int *__restrict__ idx) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int j = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (j >= m) return;
  const float *p = xyz + (size_t)b * n * 3;
  const float *q = new_xyz + ((size_t)b * m + j) * 3;
  int *o = idx + ((size_t)b * m + j) * nsample;
  const float cx = __ldg(q), cy = __ldg(q + 1), cz = __ldg(q + 2);
  int cnt = 0, first = 0;
  for (int k0 = 0; k0 < n && cnt < nsample; k0 += 32) {
    const int k = k0 + lane;
    bool hit = false;
    if (k < n) {
      const float d2 = hg_dist3_fma(cx, cy, cz, __ldg(p + (size_t)k * 3), __ldg(p + (size_t)k * 3 + 1),
                                    __ldg(p + (size_t)k * 3 + 2));
      hit = d2 < radius2;
    }
    const unsigned mask = __ballot_sync(0xffffffffu, hit);
    if (mask) {
      if (cnt == 0) first = k0 + __ffs(mask) - 1;
      const int pos = cnt + __popc(mask & ((1u << lane) - 1u));
      if (hit && pos < nsample) o[pos] = k;
      cnt += __popc(mask);
    }
  }
  if (cnt > nsample) cnt = nsample;
  const int fill = (cnt == 0) ? 0 : first;  // no hit: the reference leaves its zero-initialised row
  for (int l = cnt + lane; l < nsample; l += 32) o[l] = fill;
}

// ---- three_nn (interpolate_gpu.cu:9-59) ---------------------------------------------------------------------
__global__ void __launch_bounds__(128) three_nn_kernel(int n, int m, const float *__restrict__ unknown,
                                                       const float *__restrict__ known, float *__restrict__ dist2,
                                                       int *__restrict__ idx) {
  __shared__ float kx[512], ky[512], kz[512];
  const int b = blockIdx.y;
  const int j = blockIdx.x * 128 + threadIdx.x;
  const float *u = unknown + (size_t)b * n * 3;
  const float *kn = known + (size_t)b * m * 3;
  float ux = 0.f, uy = 0.f, uz = 0.f;
  if (j < n) {
    ux = __ldg(u + (size_t)j * 3);
    uy = __ldg(u + (size_t)j * 3 + 1);
    uz = __ldg(u + (size_t)j * 3 + 2);
  }
  // the reference keeps its running bests in double initialised to 1e40; d is a float, so comparisons are
  // the float comparisons below and an unfilled slot converts to +inf on output
  float b1 = CUDART_INF_F, b2 = CUDART_INF_F, b3 = CUDART_INF_F;
  int i1 = 0, i2 = 0, i3 = 0;
  for (int base = 0; base < m; base += 512) {
    __syncthreads();
    for (int t = threadIdx.x; t < 512 && base + t < m; t += 128) {
      kx[t] = __ldg(kn + (size_t)(base + t) * 3);
      ky[t] = __ldg(kn + (size_t)(base + t) * 3 + 1);
      kz[t] = __ldg(kn + (size_t)(base + t) * 3 + 2);
    }
    __syncthreads();
    const int lim = min(512, m - base);
    for (int t = 0; t < lim; ++t) {
      const float d = hg_dist3_fma(ux, uy, uz, kx[t], ky[t], kz[t]);
      const int k = base + t;
      if (d < b1) {
        b3 = b2; i3 = i2;
        b2 = b1; i2 = i1;
        b1 = d; i1 = k;
      } else if (d < b2) {
        b3 = b2; i3 = i2;
        b2 = d; i2 = k;
      } else if (d < b3) {
        b3 = d; i3 = k;
      }
    }
  }
  if (j < n) {
    float *o = dist2 + ((size_t)b * n + j) * 3;
    int *oi = idx + ((size_t)b * n + j) * 3;
    o[0] = b1; o[1] = b2; o[2] = b3;
    oi[0] = i1; oi[1] = i2; oi[2] = i3;
  }
}

// ---- three_interpolate (interpolate_gpu.cu:72-101): fma(p3,w3, fma(p1,w1, round(p2*w2))) -------------------
__global__ void __launch_bounds__(256) three_interpolate_kernel(int b, int c, int m, int n,
                                                                const float *__restrict__ points,
                                                                const int *__restrict__ idx,
                                                                const float *__restrict__ weight,
                                                                float *__restrict__ out) {
  const long long total = (long long)b * c * n;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(g % n);
    const long long bc = g / n;
    const int bi = (int)(bc / c);
    const int *id = idx + ((size_t)bi * n + j) * 3;
    const float *w = weight + ((size_t)bi * n + j) * 3;
    const float *p = points + (size_t)bc * m;
    out[g] = __fmaf_rn(__ldg(p + id[2]), w[2], __fmaf_rn(__ldg(p + id[0]), w[0], __fmul_rn(__ldg(p + id[1]), w[1])));
  }
}

// Staged variant: a CTA pass covers kInterpCP channels of one cloud (their m source values in shared memory), so the
// three (index, weight) pairs of an output position are loaded once for kInterpCP output rows, and the gathers hit
// shared memory.  Same arithmetic.
constexpr int kInterpCP = 8;
__global__ void __launch_bounds__(256) three_interpolate_staged_kernel(int c, int m, int n, long long groups,
                                                                       const float *__restrict__ points,
                                                                       const int *__restrict__ idx,
                                                                       const float *__restrict__ weight,
                                                                       float *__restrict__ out) {
  extern __shared__ float plane[];  // [kInterpCP][m]
  const int gpc = (c + kInterpCP - 1) / kInterpCP;
  for (long long gi = blockIdx.y; gi < groups; gi += gridDim.y) {
    const long long bi = gi / gpc;
    const int c0 = (int)(gi % gpc) * kInterpCP;
    const int nc = min(kInterpCP, c - c0);
    __syncthreads();
    for (int i = threadIdx.x; i < nc * m; i += 256) plane[i] = __ldg(points + ((size_t)bi * c + c0) * m + i);
    __syncthreads();
    for (int j = blockIdx.x * 256 + threadIdx.x; j < n; j += gridDim.x * 256) {
      const int *id = idx + ((size_t)bi * n + j) * 3;
      const float *w = weight + ((size_t)bi * n + j) * 3;
      const int i0 = id[0], i1 = id[1], i2 = id[2];
      const float w0 = w[0], w1 = w[1], w2 = w[2];
#pragma unroll
      for (int q = 0; q < kInterpCP; ++q)
        if (q < nc) {
          const float *p = plane + q * m;
          out[((size_t)bi * c + c0 + q) * n + j] = __fmaf_rn(p[i2], w2, __fmaf_rn(p[i0], w0, __fmul_rn(p[i1], w1)));
        }
    }
  }
}

// ---- furthest point sampling ---------------------------------------------------------------------------------
// POLICY_P2   : sampling_gpu.cu:69-173.  d = fma(dz,dz,fma(dx,dx,dy*dy)); points with |p|^2 <= 1e-3 are skipped;
//               start index 0; ties resolved like the reference's shared-memory tree: smallest
//               (bitreverse(k mod bs), k) where bs = opt_n_threads(n).
// POLICY_TORCH: model/pointnet2_utils.py:63-84.  d = (dx*dx + dy*dy) + dz*dz (no FMA); every point is a
//               candidate; start index given; torch.max tie rule = lowest index.
enum { POLICY_P2 = 0, POLICY_TORCH = 1 };

// TH threads per cloud: 256 up to 4096 points, 1024 beyond (the register-resident cloud stays <= 16 points/thread
// up to 16384 points; the per-round cost is PPT distance updates + one 64-bit block max)
template <int POLICY, int PPT, int TH, typename IdxT>
__global__ void __launch_bounds__(TH) fps_kernel(const float *__restrict__ dataset_all, int n, int m,
                                                          int log2bs, const long long *__restrict__ start,
                                                          IdxT *__restrict__ idxs_all) {
  constexpr int W = TH / 32;
  __shared__ unsigned long long wbest[2][W];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *dataset = dataset_all + (size_t)b * n * 3;
  IdxT *idxs = idxs_all + (size_t)b * m;
  const int bs = 1 << log2bs;
  const unsigned R = (unsigned)((n + bs - 1) >> log2bs);

  float px[PPT], py[PPT], pz[PPT], td[PPT];
  unsigned low[PPT];  // ~tie-composite; 0 marks a point that can never be selected
#pragma unroll
  for (int r = 0; r < PPT; ++r) {
    const int k = tid + r * TH;
    px[r] = py[r] = pz[r] = 0.f;
    td[r] = 1e10f;
    low[r] = 0u;
    if (k < n) {
      px[r] = __ldg(dataset + (size_t)k * 3);
      py[r] = __ldg(dataset + (size_t)k * 3 + 1);
      pz[r] = __ldg(dataset + (size_t)k * 3 + 2);
      unsigned comp;
      bool valid = true;
      if (POLICY == POLICY_P2) {
        const float mag = __fmaf_rn(pz[r], pz[r], __fmaf_rn(px[r], px[r], __fmul_rn(py[r], py[r])));
        valid = !((double)mag <= 1e-3);
        const unsigned tb = (unsigned)k & (unsigned)(bs - 1);
        const unsigned rev = log2bs ? (__brev(tb) >> (32 - log2bs)) : 0u;
        comp = rev * R + ((unsigned)k >> log2bs);
      } else {
        comp = (unsigned)k;
      }
      low[r] = valid ? ~comp : 0u;
    }
  }
  // One round = distance update of the register-resident points, then a block-wide lexicographic maximum of
  // (distance bits, tie composite) with the winner's COORDINATES travelling with its key: the round's critical path has
  // no dependent global load and no index decode (the raw composites are decoded by all threads after the last round).
  // The round is one latency chain, so it is kept shallow (tools/ubench/redux_latency.cu on a B200: CREDUX round trip
  // 27 cycles, a 64-bit shuffle butterfly 195, BAR.SYNC 21, dependent LDS 43): per level, a max tree + CREDUX over the
  // distance bits, then the same over the composites of the entries that hold that distance, then predicated moves;
  // clouds up to 2048 points run on one warp per scheduler.  A point that can never be selected has composite 0 and
  // distance 0 for ever ("nothing" = composite 0).
  static_assert(W <= 32, "one lane per warp in the second reduction level");
  __shared__ float4 wcoord[2][W];
#pragma unroll
  for (int r = 0; r < PPT; ++r)
    if (!low[r]) td[r] = 0.f;
  int old = (POLICY == POLICY_P2) ? 0 : (int)start[b];
  if (tid == 0) idxs[0] = (IdxT)old;
  float x1 = __ldg(dataset + (size_t)old * 3), y1 = __ldg(dataset + (size_t)old * 3 + 1),
        z1 = __ldg(dataset + (size_t)old * 3 + 2);
  for (int j = 1; j < m; ++j) {
    unsigned t[PPT];
#pragma unroll
    for (int r = 0; r < PPT; ++r) {
      float d;
      if (POLICY == POLICY_P2) {
        d = hg_dist3_fma(px[r], py[r], pz[r], x1, y1, z1);
      } else {
        const float dx = __fsub_rn(px[r], x1), dy = __fsub_rn(py[r], y1), dz = __fsub_rn(pz[r], z1);
        d = __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
      }
      td[r] = fminf(d, td[r]);
      t[r] = __float_as_uint(td[r]);  // distances are >= 0: their bit patterns order like unsigned integers
    }
#pragma unroll
    for (int s = 1; s < PPT; s <<= 1)
#pragma unroll
      for (int r = 0; r + s < PPT; r += 2 * s) t[r] = max(t[r], t[r + s]);
    const unsigned whi = __reduce_max_sync(0xffffffffu, t[0]);
#pragma unroll
    for (int r = 0; r < PPT; ++r) t[r] = __float_as_uint(td[r]) == whi ? low[r] : 0u;
#pragma unroll
    for (int s = 1; s < PPT; s <<= 1)
#pragma unroll
      for (int r = 0; r + s < PPT; r += 2 * s) t[r] = max(t[r], t[r + s]);
    const unsigned wlo = __reduce_max_sync(0xffffffffu, t[0]);
    // one lane per warp: the composites are distinct; a warp with nothing to offer writes composite 0 from lane 0
    if (t[0] == wlo && (wlo != 0u || lane == 0)) {
      float bx = 0.f, by = 0.f, bz = 0.f;
#pragma unroll
      for (int r = 0; r < PPT; ++r)
        if (__float_as_uint(td[r]) == whi && low[r] == wlo) {
          bx = px[r];
          by = py[r];
          bz = pz[r];
        }
      wbest[j & 1][warp] = ((unsigned long long)whi << 32) | wlo;
      wcoord[j & 1][warp] = make_float4(bx, by, bz, 0.f);
    }
    __syncthreads();
    unsigned ahi, alo;
    float4 c;
    if (W <= 8) {  // few warps: every thread reads all (key, coordinates) pairs at once
      unsigned long long k[W];
      float4 kc[W];
#pragma unroll
      for (int w = 0; w < W; ++w) {
        k[w] = wbest[j & 1][w];
        kc[w] = wcoord[j & 1][w];
      }
      ahi = 0u;
#pragma unroll
      for (int w = 0; w < W; ++w) ahi = max(ahi, (unsigned)(k[w] >> 32));
      alo = 0u;
#pragma unroll
      for (int w = 0; w < W; ++w) alo = max(alo, (unsigned)(k[w] >> 32) == ahi ? (unsigned)k[w] : 0u);
      c = kc[0];
#pragma unroll
      for (int w = 1; w < W; ++w)
        if ((unsigned)(k[w] >> 32) == ahi && (unsigned)k[w] == alo) c = kc[w];
    } else {
      const unsigned long long mine = lane < W ? wbest[j & 1][lane] : 0ull;
      const unsigned mhi = (unsigned)(mine >> 32), mlo = (unsigned)mine;
      ahi = __reduce_max_sync(0xffffffffu, mhi);
      alo = __reduce_max_sync(0xffffffffu, mhi == ahi ? mlo : 0u);
      const int wwin = __ffs(__ballot_sync(0xffffffffu, lane < W && mhi == ahi && mlo == alo)) - 1;
      c = wcoord[j & 1][wwin];
    }
    if (alo == 0u) {  // no selectable point at all: the reference keeps writing index 0
      x1 = __ldg(dataset);
      y1 = __ldg(dataset + 1);
      z1 = __ldg(dataset + 2);
    } else {
      x1 = c.x;
      y1 = c.y;
      z1 = c.z;
    }
    if (tid == 0) idxs[j] = (IdxT)(alo == 0u ? 0xffffffffu : ~alo);  // raw composite, decoded below
  }
  __syncthreads();
  for (int j = 1 + tid; j < m; j += TH) {
    const unsigned comp = (unsigned)idxs[j];
    int out = 0;
    if (comp != 0xffffffffu) {
      if (POLICY == POLICY_P2) {
        const unsigned rev = comp / R, rr = comp % R;
        const unsigned tb = log2bs ? (__brev(rev) >> (32 - log2bs)) : 0u;
        out = (int)(tb + (rr << log2bs));
      } else {
        out = (int)comp;
      }
    }
    idxs[j] = (IdxT)out;
  }
}

template <int POLICY, typename IdxT>
int launch_fps(const float *dataset, int b, int n, int m, const long long *start, IdxT *idxs, cudaStream_t stream) {
  int log2bs = 0;
  if (POLICY == POLICY_P2) {
    const int bs = ref_opt_n_threads(n);
    while ((1 << log2bs) < bs) ++log2bs;
  }
  // threads per cloud: the round is a latency chain (update -> warp max -> barrier -> block max), so small clouds run
  // on ONE warp per scheduler (128 threads, <= 8 points per thread) and do not contend for issue slots
  const int th = n > 4096 ? 1024 : (n > 2048 ? 256 : 128);
  const int ppt = (n + th - 1) / th;
#define HG_FPS_CASE(P, TH)                                                                                \
  if (th == TH && ppt <= P) {                                                                             \
    const bool prof = hg_prof_begin(HG_PROF_FPS, stream);                                                 \
    fps_kernel<POLICY, P, TH, IdxT><<<b, TH, 0, stream>>>(dataset, n, m, log2bs, start, idxs);            \
    hg_prof_end(HG_PROF_FPS, stream, prof);                                                               \
    HG_CHECK_LAUNCH("fps_kernel");                                                                        \
    return HG_OK;                                                                                         \
  }
  HG_FPS_CASE(1, 128)
  HG_FPS_CASE(2, 128)
  HG_FPS_CASE(4, 128)
  HG_FPS_CASE(8, 128)
  HG_FPS_CASE(16, 128)
  HG_FPS_CASE(16, 256)
  HG_FPS_CASE(8, 1024)
  HG_FPS_CASE(16, 1024)
  HG_FPS_CASE(32, 1024)
  HG_FPS_CASE(64, 1024)
#undef HG_FPS_CASE
  hg_set_error("fps: n=%d > 65536 points per cloud unsupported", n);
  return HG_E_UNSUPPORTED;
}

}  // namespace

// ================================================ C ABI =====================================================
HG_API int hg_p2_gather_points(int b, int c, int n, int npoints, const float *points, const int *idx, float *out,
                               hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_gather_points");
  HG_REQUIRE(points && idx && out, HG_E_BADARG, "gather_points: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && n > 0 && npoints > 0, HG_E_BADARG, "gather_points: sizes must be positive");
  return launch_gather(points, idx, b, c, n, npoints, out, hg_stream(stream_), -1);
}

HG_API size_t hg_p2_scatter_workspace_bytes(int b, int n, int nedges) {
  if (b <= 0 || n <= 0 || nedges <= 0) return 0;
  return hg_csr_stable_workspace_bytes(b, n, nedges);
}

HG_API int hg_p2_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out, const int *idx,
                                    float *grad_points, void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_gather_points_grad");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && grad_points, HG_E_BADARG, "gather_points_grad: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && n > 0 && npoints > 0, HG_E_BADARG, "gather_points_grad: sizes must be positive");
  HgCsr csr;
  int rc = hg_csr_build(idx, b, npoints, n, workspace, workspace_bytes, &csr, stream);
  if (rc) return rc;
  rc = launch_scatter_unweighted(grad_out, csr, b, c, n, npoints, grad_points, stream);
  if (rc) return rc;
  HG_CHECK_LAUNCH("gather_points_grad");
  return HG_OK;
}

HG_API int hg_p2_furthest_point_sampling(int b, int n, int m, const float *dataset, float *temp, int *idxs,
                                         hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_furthest_point_sampling");
  (void)temp;  // the reference's global scratch (sampling.cpp:74-76); distances live in registers here
  HG_REQUIRE(dataset && idxs, HG_E_BADARG, "furthest_point_sampling: null pointer");
  HG_REQUIRE(b > 0 && n > 0 && m >= 0, HG_E_BADARG, "furthest_point_sampling: bad sizes");
  if (m == 0) return HG_OK;
  return launch_fps<POLICY_P2, int>(dataset, b, n, m, nullptr, idxs, hg_stream(stream_));
}

HG_API int hg_fps_torch_f32(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *centroids,
                            hgStream stream_) {
  HG_NVTX_RANGE("hg_fps_torch_f32");
  HG_REQUIRE(xyz && start && centroids, HG_E_BADARG, "fps_torch: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && npoint >= 0, HG_E_BADARG, "fps_torch: bad sizes");
  if (npoint == 0) return HG_OK;
  return launch_fps<POLICY_TORCH, long long>(xyz, B, N, npoint, (const long long *)start, (long long *)centroids,
                                             hg_stream(stream_));
}

HG_API int hg_p2_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz, const float *xyz,
                            int *idx, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_ball_query");
  HG_REQUIRE(new_xyz && xyz && idx, HG_E_BADARG, "ball_query: null pointer");
  HG_REQUIRE(b > 0 && n > 0 && m > 0 && nsample > 0, HG_E_BADARG, "ball_query: sizes must be positive");
  HG_REQUIRE(b <= 65535, HG_E_UNSUPPORTED, "ball_query: b=%d > 65535", b);
  const float radius2 = radius * radius;  // ball_query_gpu.cu:22 (FMUL)
  ball_query_kernel<<<dim3((m + 3) / 4, b), 128, 0, hg_stream(stream_)>>>(n, m, radius2, nsample, new_xyz, xyz, idx);
  HG_CHECK_LAUNCH("ball_query");
  return HG_OK;
}

HG_API int hg_p2_group_points(int b, int c, int n, int npoints, int nsample, const float *points, const int *idx,
                              float *out, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_group_points");
  HG_REQUIRE(points && idx && out, HG_E_BADARG, "group_points: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && n > 0 && npoints > 0 && nsample > 0, HG_E_BADARG, "group_points: sizes must be positive");
  return launch_gather(points, idx, b, c, n, npoints * nsample, out, hg_stream(stream_), HG_PROF_GROUP);
}

// pointnet2_utils.py:279-333 QueryAndGroup.forward after its ball query, written once: rows 0..2 = grouped_xyz -
// new_xyz, rows 3.. = grouped features (the reference: two grouping ops, an in-place subtraction and a torch.cat)
HG_API int hg_p2_group_concat(int b, int c, int n, int npoints, int nsample, const float *xyz, const float *new_xyz,
                              const float *features, const int *idx, float *out, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_group_concat");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(xyz && new_xyz && idx && out, HG_E_BADARG, "group_concat: null pointer");
  HG_REQUIRE(b > 0 && c >= 0 && n > 0 && npoints > 0 && nsample > 0, HG_E_BADARG, "group_concat: bad sizes");
  HG_REQUIRE(c == 0 || features, HG_E_BADARG, "group_concat: features is null but c > 0");
  const long long total = (long long)b * npoints * nsample;
  group_xyz_rel_kernel<<<hg_grid_for(total, 256, 32), 256, 0, stream>>>(xyz, new_xyz, idx, n, npoints, nsample, 3 + c, total,
                                                                        out);
  HG_CHECK_LAUNCH("group_xyz_rel_kernel");
  if (c > 0) return launch_gather(features, idx, b, c, n, npoints * nsample, out, stream, HG_PROF_GROUP, 3 + c, 3);
  return HG_OK;
}

// backward of hg_p2_group_concat w.r.t. the features (b,c,n) and the coordinates (as (b,3,n), channel-major); either
// output may be NULL.  (d/d new_xyz is minus the sum over the samples of rows 0..2: a plain reduction, left to the host.)
HG_API int hg_p2_group_concat_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out, const int *idx,
                                   float *grad_xyz_t, float *grad_features, void *workspace, size_t workspace_bytes,
                                   hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_group_concat_grad");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && (grad_xyz_t || grad_features), HG_E_BADARG, "group_concat_grad: null pointer");
  HG_REQUIRE(b > 0 && c >= 0 && n > 0 && npoints > 0 && nsample > 0, HG_E_BADARG, "group_concat_grad: bad sizes");
  const int E = npoints * nsample;
  HgCsr csr;
  int rc = hg_csr_build(idx, b, E, n, workspace, workspace_bytes, &csr, stream);
  if (rc) return rc;
  if (grad_xyz_t) {
    rc = launch_scatter_unweighted(grad_out, csr, b, 3, n, E, grad_xyz_t, stream, 3 + c, 0);
    if (rc) return rc;
    HG_CHECK_LAUNCH("group_concat_grad(xyz)");
  }
  if (grad_features && c > 0) {
    rc = launch_scatter_unweighted(grad_out, csr, b, c, n, E, grad_features, stream, 3 + c, 3);
    if (rc) return rc;
    HG_CHECK_LAUNCH("group_concat_grad(features)");
  }
  return HG_OK;
}

HG_API int hg_p2_group_points_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out,
                                   const int *idx, float *grad_points, void *workspace, size_t workspace_bytes,
                                   hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_group_points_grad");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && grad_points, HG_E_BADARG, "group_points_grad: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && n > 0 && npoints > 0 && nsample > 0, HG_E_BADARG,
             "group_points_grad: sizes must be positive");
  const int E = npoints * nsample;
  HgCsr csr;
  int rc = hg_csr_build(idx, b, E, n, workspace, workspace_bytes, &csr, stream);
  if (rc) return rc;
  rc = launch_scatter_unweighted(grad_out, csr, b, c, n, E, grad_points, stream);
  if (rc) return rc;
  HG_CHECK_LAUNCH("group_points_grad");
  return HG_OK;
}

HG_API int hg_p2_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int *idx,
                          hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_three_nn");
  HG_REQUIRE(unknown && known && dist2 && idx, HG_E_BADARG, "three_nn: null pointer");
  HG_REQUIRE(b > 0 && n > 0 && m > 0, HG_E_BADARG, "three_nn: sizes must be positive");
  HG_REQUIRE(b <= 65535, HG_E_UNSUPPORTED, "three_nn: b=%d > 65535", b);
  three_nn_kernel<<<dim3((n + 127) / 128, b), 128, 0, hg_stream(stream_)>>>(n, m, unknown, known, dist2, idx);
  HG_CHECK_LAUNCH("three_nn");
  return HG_OK;
}

HG_API int hg_p2_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx,
                                   const float *weight, float *out, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_three_interpolate");
  HG_REQUIRE(points && idx && weight && out, HG_E_BADARG, "three_interpolate: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && m > 0 && n > 0, HG_E_BADARG, "three_interpolate: sizes must be positive");
  const size_t smem = (size_t)kInterpCP * m * sizeof(float);
  if (smem <= 96 * 1024) {
    if (smem > 48 * 1024)
      HG_CUDA(cudaFuncSetAttribute(three_interpolate_staged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long groups = (long long)b * ((c + kInterpCP - 1) / kInterpCP);
    int gx = (n + 255) / 256;
    long long gx_cap = (8LL * hg_sm_count() + groups - 1) / groups;
    if (gx_cap < 1) gx_cap = 1;
    if (gx > gx_cap) gx = (int)gx_cap;
    three_interpolate_staged_kernel<<<dim3(gx, (unsigned)(groups < 65535 ? groups : 65535)), 256, smem, hg_stream(stream_)>>>(
        c, m, n, groups, points, idx, weight, out);
  } else {
    const long long total = (long long)b * c * n;
    three_interpolate_kernel<<<hg_grid_for(total, 256, 32), 256, 0, hg_stream(stream_)>>>(b, c, m, n, points, idx, weight, out);
  }
  HG_CHECK_LAUNCH("three_interpolate");
  return HG_OK;
}

HG_API int hg_p2_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int *idx,
                                        const float *weight, float *grad_points, void *workspace,
                                        size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_p2_three_interpolate_grad");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && weight && grad_points, HG_E_BADARG, "three_interpolate_grad: null pointer");
  HG_REQUIRE(b > 0 && c > 0 && m > 0 && n > 0, HG_E_BADARG, "three_interpolate_grad: sizes must be positive");
  HgCsr csr;
  int rc = hg_csr_build(idx, b, n * 3, m, workspace, workspace_bytes, &csr, stream);
  if (rc) return rc;
  const long long total = (long long)b * c * m;
  scatter_channel_major_kernel<3, true><<<hg_grid_for(total, 256, 32), 256, 0, stream>>>(grad_out, weight, csr.off, csr.list, b,
                                                                                         c, m, n * 3, grad_points);
  HG_CHECK_LAUNCH("three_interpolate_grad");
  return HG_OK;
}
