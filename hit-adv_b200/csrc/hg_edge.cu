// hg_edge.cu -- DGCNN edge features (model/dgcnn_cls.py:16-43 get_graph_feature), forward and backward.
//
//   out[b, c,     n, t] = x[b, c, idx[b,n,t]] - x[b, c, n]          c < C
//   out[b, C + c, n, t] = x[b, c, n]
//
// The reference builds this with an index gather on a transposed copy, a k-fold `repeat`, a `cat` and a
// `permute(...).contiguous()`: four full-size [B,N,k,2C] tensors are written and re-read (671 MB each at
// B=32, C=128, N=1024, k=20) and autograd keeps two of them.  Here the output is written once, straight in its final
// layout; nothing else of that size exists.  HBM-bound: algorithmic bytes = the output (8 B per edge per channel
// forward; backward reads the same amount once).
//
// Backward:  grad_x[b,c,n] = sum_t (g[b,C+c,n,t] - g[b,c,n,t])  +  sum_{(m,t): idx[b,m,t] = n} g[b,c,m,t]
// The reference's second sum is an `index_put_(accumulate=True)` with floating-point atomics (run-to-run rounding
// differences); here it is a walk over a CSR reverse map in ascending edge order: deterministic.
#include "hg_common.cuh"

namespace {

// ---- forward: a CTA pass covers kEdgeCP channels of one cloud: their N source values are staged in shared memory
// and every index load (the expensive part: 8 B per edge, L2) serves kEdgeCP x 2 output rows ----------------------
// Larger clouds stage fewer planes per pass (kEdgeCP = 2 up to 25600 points, 1 up to 51200); beyond that the pass reads
// its four planes from x through L2 (STAGED = false), as the backward's unstaged variant does.
template <int kEdgeCP, bool STAGED, bool VEC4>
__global__ void __launch_bounds__(256) edge_feature_kernel(const float *__restrict__ x,
                                                           const long long *__restrict__ idx, int C, int N, int k,
                                                           long long groups, float *__restrict__ out) {
  extern __shared__ float smem_planes[];  // STAGED: [kEdgeCP][N]
  const int E = N * k;
  const int gpc = (C + kEdgeCP - 1) / kEdgeCP;  // channel groups per cloud
  for (long long gi = blockIdx.y; gi < groups; gi += gridDim.y) {
    const long long b = gi / gpc;
    const int c0 = (int)(gi % gpc) * kEdgeCP;
    const int nc = min(kEdgeCP, C - c0);
    const long long *id = idx + (size_t)b * E;
    const float *plane = STAGED ? smem_planes : x + ((size_t)b * C + c0) * N;
    if (STAGED) {
      __syncthreads();
      for (int i = threadIdx.x; i < nc * N; i += 256) smem_planes[i] = __ldg(x + ((size_t)b * C + c0) * N + i);
      __syncthreads();
    }
    float *dstA = out + ((size_t)b * 2 * C + c0) * E;
    float *dstB = dstA + (size_t)C * E;
    if (VEC4) {  // k % 4 == 0: the four edges of a float4 share their centre point
      for (int e = (blockIdx.x * 256 + threadIdx.x) * 4; e < E; e += gridDim.x * 1024) {
        const longlong2 i01 = *reinterpret_cast<const longlong2 *>(id + e);
        const longlong2 i23 = *reinterpret_cast<const longlong2 *>(id + e + 2);
        const int n = e / k;
#pragma unroll
        for (int q = 0; q < kEdgeCP; ++q) {
          if (q < nc) {
            const float *pl = plane + q * N;
            const float ctr = pl[n];
            float4 a;
            a.x = pl[i01.x] - ctr;
            a.y = pl[i01.y] - ctr;
            a.z = pl[i23.x] - ctr;
            a.w = pl[i23.y] - ctr;
            __stcs(reinterpret_cast<float4 *>(dstA + (size_t)q * E + e), a);  // streaming: consumed by the next layer
            __stcs(reinterpret_cast<float4 *>(dstB + (size_t)q * E + e), make_float4(ctr, ctr, ctr, ctr));
          }
        }
      }
    } else {
      for (int e = blockIdx.x * 256 + threadIdx.x; e < E; e += gridDim.x * 256) {
        const long long ii = id[e];
        const int n = e / k;
        for (int q = 0; q < nc; ++q) {
          // unstaged, N may reach 2^31 / k, so q * N is taken in 64 bits (staged, q * N < 51200 * 4)
          const float ctr = STAGED ? plane[q * N + n] : plane[(size_t)q * N + n];
          dstA[(size_t)q * E + e] = (STAGED ? plane[q * N + ii] : plane[(size_t)q * N + ii]) - ctr;
          dstB[(size_t)q * E + e] = ctr;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) edge_keys_kernel(const long long *__restrict__ idx, long long total, int N,
                                                        int *__restrict__ keys) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long a = idx[g];
    keys[g] = (a >= 0 && a < N) ? (int)a : -1;
  }
}

// ---- backward: one CTA per (b,c) plane.  Thread n streams row n of both halves (k contiguous floats: a warp
// covers 32*k contiguous floats), keeps sum_t (gB - gA) in a register and parks the gA row in shared memory; after
// a barrier the incoming edges are summed from shared memory in ascending edge order.
constexpr int kHubSplit = 32;
constexpr int kGradThreads = 512;  // two CTAs of 512 per SM (80 KB of shared memory each at N*k = 20480): the three
                                   // dependent phases of a plane are latency-bound, so more rows in flight per phase
template <bool STAGED>
__global__ void __launch_bounds__(kGradThreads) edge_feature_grad_kernel(const float *__restrict__ g,
                                                                const int *__restrict__ off,
                                                                const int *__restrict__ list, int C, int N, int k,
                                                                long long planes, float *__restrict__ grad_x) {
  extern __shared__ float sA[];  // STAGED: [N*k] the gA plane
  const int E = N * k;
  const bool vec = (k & 3) == 0;
  for (long long bc = blockIdx.x; bc < planes; bc += gridDim.x) {
    const long long b = bc / C;
    const int c = (int)(bc % C);
    const float *gA = g + ((size_t)b * 2 * C + c) * E;
    const float *gB = gA + (size_t)C * E;
    const int *o = off + (size_t)b * (N + 1);
    const int *l = list + (size_t)b * E;
    float *dst = grad_x + (size_t)bc * N;
    __syncthreads();
    for (int n0 = 0; n0 < N; n0 += kGradThreads) {
      const int n = n0 + threadIdx.x;
      float own = 0.f;
      if (n < N) {
        const float *ra = gA + (size_t)n * k, *rb = gB + (size_t)n * k;
        if (vec) {
          for (int t = 0; t < k; t += 4) {
            const float4 a = __ldcs(reinterpret_cast<const float4 *>(ra + t));
            const float4 bb = __ldcs(reinterpret_cast<const float4 *>(rb + t));
            own += (bb.x - a.x);
            own += (bb.y - a.y);
            own += (bb.z - a.z);
            own += (bb.w - a.w);
            if (STAGED) *reinterpret_cast<float4 *>(sA + (size_t)n * k + t) = a;
          }
        } else {
          for (int t = 0; t < k; ++t) {
            const float a = ra[t];
            own += (rb[t] - a);
            if (STAGED) sA[(size_t)n * k + t] = a;
          }
        }
      }
      if (!STAGED && n < N) {  // plane too large for shared memory: gather from global (L2)
        float acc = own;
        for (int q = o[n]; q < o[n + 1]; ++q) acc += gA[l[q]];
        dst[n] = acc;
      }
      if (STAGED && n < N) dst[n] = own;  // finished below
    }
    if (STAGED) {
      // kNN graphs of learned features have hubs (in-degrees in the hundreds next to a mean of k): a thread sums at most
      // kHubSplit incoming edges of its point; what is left of a hub is summed by a whole warp afterwards (lanes
      // stride the rest of the segment, fixed-order tree) -- same bits on every run, no lane waits for a hub.
      int *hubq = reinterpret_cast<int *>(sA + E);  // [N] points with more than kHubSplit incoming edges
      __shared__ int nhub;
      if (threadIdx.x == 0) nhub = 0;
      __syncthreads();
      for (int n = threadIdx.x; n < N; n += kGradThreads) {
        float acc = dst[n];
        const int q1 = o[n + 1];
        int q = o[n];
        const int qe = min(q1, q + kHubSplit);
        for (; q + 3 < qe; q += 4) {  // four list entries in flight
          const int e0 = __ldg(l + q), e1 = __ldg(l + q + 1), e2 = __ldg(l + q + 2), e3 = __ldg(l + q + 3);
          acc += sA[e0];
          acc += sA[e1];
          acc += sA[e2];
          acc += sA[e3];
        }
        for (; q < qe; ++q) acc += sA[__ldg(l + q)];
        dst[n] = acc;
        if (q1 > qe) hubq[atomicAdd(&nhub, 1)] = n;
      }
      __syncthreads();
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      for (int h = warp; h < nhub; h += kGradThreads / 32) {
        const int n = hubq[h];
        const int q1 = o[n + 1];
        float part = 0.f;
        for (int q = o[n] + kHubSplit + lane; q < q1; q += 32) part += sA[__ldg(l + q)];
#pragma unroll
        for (int st = 16; st > 0; st >>= 1) part += __shfl_down_sync(0xffffffffu, part, st);
        if (lane == 0) dst[n] += part;
      }
    }
  }
}

constexpr size_t kEdgeStageBytes = 200 * 1024;  // shared memory a forward CTA may stage its planes in

template <int kEdgeCP, bool STAGED>
int edge_feature_launch(const float *x, const int64_t *idx, int B, int C, int N, int k, float *out, cudaStream_t stream) {
  const long long groups = (long long)B * ((C + kEdgeCP - 1) / kEdgeCP);
  const int E = N * k;
  const bool vec = (k % 4 == 0) && ((reinterpret_cast<uintptr_t>(idx) | reinterpret_cast<uintptr_t>(out)) % 16 == 0);
  const int per_block = vec ? 1024 : 256;
  int gx = (E + per_block - 1) / per_block;
  // enough CTAs to fill the machine a few times over, each amortising its plane staging over >= 1/gx of the edges
  int gx_cap = (int)((8LL * hg_sm_count() + groups - 1) / groups);
  if (gx_cap < 1) gx_cap = 1;
  if (gx > gx_cap) gx = gx_cap;
  const int gy = (int)(groups < 65535 ? groups : 65535);
  const size_t smem = STAGED ? (size_t)kEdgeCP * N * sizeof(float) : 0;
  const bool prof = hg_prof_begin(HG_PROF_GROUP, stream);
  if (vec) {
    if (smem > 48 * 1024)
      HG_CUDA((cudaFuncSetAttribute(edge_feature_kernel<kEdgeCP, STAGED, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)));
    edge_feature_kernel<kEdgeCP, STAGED, true><<<dim3(gx, gy), 256, smem, stream>>>(x, (const long long *)idx, C, N, k, groups, out);
  } else {
    if (smem > 48 * 1024)
      HG_CUDA((cudaFuncSetAttribute(edge_feature_kernel<kEdgeCP, STAGED, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)));
    edge_feature_kernel<kEdgeCP, STAGED, false><<<dim3(gx, gy), 256, smem, stream>>>(x, (const long long *)idx, C, N, k, groups, out);
  }
  hg_prof_end(HG_PROF_GROUP, stream, prof);
  HG_CHECK_LAUNCH("edge_feature_kernel");
  return HG_OK;
}

}  // namespace

// dgcnn_cls.py:16-43 (feature build only; the neighbour search is hg_knn_self_f32 / model_seams.knn)
HG_API int hg_edge_feature_f32(const float *x, const int64_t *idx, int B, int C, int N, int k, float *out,
                               hgStream stream_) {
  HG_NVTX_RANGE("hg_edge_feature_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(x && idx && out, HG_E_BADARG, "edge_feature: null pointer");
  HG_REQUIRE(B > 0 && C > 0 && N > 0 && k > 0, HG_E_BADARG, "edge_feature: sizes must be positive");
  HG_REQUIRE((long long)N * k < (1LL << 31), HG_E_UNSUPPORTED, "edge_feature: N*k too large");
  const size_t plane = (size_t)N * sizeof(float);
  if (4 * plane <= kEdgeStageBytes) return edge_feature_launch<4, true>(x, idx, B, C, N, k, out, stream);
  if (2 * plane <= kEdgeStageBytes) return edge_feature_launch<2, true>(x, idx, B, C, N, k, out, stream);
  if (plane <= kEdgeStageBytes) return edge_feature_launch<1, true>(x, idx, B, C, N, k, out, stream);
  return edge_feature_launch<4, false>(x, idx, B, C, N, k, out, stream);
}

HG_API size_t hg_edge_feature_grad_workspace_bytes(int B, int N, int k) {
  if (B <= 0 || N <= 0 || k <= 0) return 0;
  return hg_layout_bytes<HgKeysCsr>(B, N, (long long)N * k, true);
}

HG_API int hg_edge_feature_grad_f32(const float *grad_out, const int64_t *idx, int B, int C, int N, int k,
                                    float *grad_x, void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_edge_feature_grad_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && grad_x, HG_E_BADARG, "edge_feature_grad: null pointer");
  HG_REQUIRE(B > 0 && C > 0 && N > 0 && k > 0, HG_E_BADARG, "edge_feature_grad: sizes must be positive");
  HG_REQUIRE((long long)N * k < (1LL << 31), HG_E_UNSUPPORTED, "edge_feature_grad: N*k too large");
  HG_REQUIRE(workspace && workspace_bytes >= hg_edge_feature_grad_workspace_bytes(B, N, k), HG_E_WORKSPACE,
             "edge_feature_grad: workspace too small");
  const int E = N * k;
  const auto w = hg_layout_at<HgKeysCsr>(workspace, B, N, (long long)E, true);
  const long long te = (long long)B * E;
  edge_keys_kernel<<<hg_grid_for(te, 256, 32), 256, 0, stream>>>((const long long *)idx, te, N, w.keys);
  HG_CHECK_LAUNCH("edge_keys_kernel");
  HgCsr csr;
  // stable build (ascending edge order inside every segment): kNN graphs of high-dimensional features have hubs
  // with in-degrees in the hundreds, which rules out the unordered build + O(deg^2) ordered walk used elsewhere
  int rc = hg_csr_build(w.keys, B, E, N, w.csr.ptr, w.csr.bytes, &csr, stream);
  if (rc) return rc;
  const long long planes = (long long)B * C;
  const size_t smem = ((size_t)E + (size_t)N) * sizeof(float);  // gA plane + hub queue
  const bool staged = smem <= 200 * 1024;
  long long grid = planes;
  const long long cap = (long long)hg_sm_count() * 8;
  if (grid > cap) grid = cap;
  if (staged) {
    if (smem > 48 * 1024)
      HG_CUDA(cudaFuncSetAttribute(edge_feature_grad_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    edge_feature_grad_kernel<true><<<(int)grid, kGradThreads, smem, stream>>>(grad_out, csr.off, csr.list, C, N, k, planes, grad_x);
  } else {
    edge_feature_grad_kernel<false><<<(int)grid, kGradThreads, 0, stream>>>(grad_out, csr.off, csr.list, C, N, k, planes, grad_x);
  }
  HG_CHECK_LAUNCH("edge_feature_grad_kernel");
  return HG_OK;
}
