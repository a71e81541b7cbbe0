// hg_seams.cu -- the torch-level geometry functions the PointNet++ SSG victim calls inside its forward
// (model/pointnet2_utils.py:19-107): square_distance, query_ball_point, index_points (+ backward).
// (farthest_point_sample lives in hg_pointnet2.cu next to the pointnet2_ops FPS it shares a kernel with.)
//
// Reference arithmetic, restated bit-exactly (SURVEY.md section 8 a-bis):
//   square_distance: d[n,m] = ((-2*zz_nm) + rs_n) + rd_m, zz = FMA chain (torch.matmul), rs/rd = torch.sum(x**2,-1)
//   query_ball_point: keep d <= float32(radius**2) ("group_idx[sqrdists > radius**2] = N"), ascending index,
//                     first nsample, pad with the first; the reference gets there by SORTING a [B,S,N] int64
//                     tensor (268 MB at B=64,S=512,N=1024) -- here it is one ballot-compacted scan.
#include "hg_common.cuh"

namespace {

__device__ __forceinline__ float sumsq_cascade(const float *a, int C) {
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
  for (int c = 0; c < C; ++c) {
    acc0 = __fadd_rn(acc0, __fmul_rn(a[c], a[c]));
    if (((c + 1) & 15) == 0) {
      acc1 = __fadd_rn(acc1, acc0);
      acc0 = 0.f;
      if (((c + 1) & 255) == 0) {
        acc2 = __fadd_rn(acc2, acc1);
        acc1 = 0.f;
      }
    }
  }
  return __fadd_rn(__fadd_rn(acc0, acc1), acc2);
}

// A CTA owns (b, 32 source rows, 1024 target columns): every thread keeps its four target points (and their squared
// norms) in registers and walks the 32 source rows staged in shared memory -- one float4 store per row, no integer
// division, each input read once per CTA; HBM-bound on the [B,N,M] output.  C <= 8 (the model calls it with C = 3);
// wider features take the generic kernel below.
constexpr int kSqRows = 32, kSqMaxC = 8;
__global__ void __launch_bounds__(256) square_distance_small_c_kernel(const float *__restrict__ src,
                                                                      const float *__restrict__ dst, int N, int M,
                                                                      int C, float *__restrict__ out) {
  __shared__ float srow[kSqRows][kSqMaxC + 1];  // [row][c], last = squared norm
  const int b = blockIdx.z, n0 = blockIdx.y * kSqRows;
  for (int t = threadIdx.x; t < kSqRows; t += 256) {
    const int n = n0 + t;
    if (n < N) {
      const float *sp = src + ((size_t)b * N + n) * C;
      for (int c = 0; c < C; ++c) srow[t][c] = sp[c];
      srow[t][kSqMaxC] = sumsq_cascade(sp, C);
    }
  }
  const int m0 = (blockIdx.x * 256 + threadIdx.x) * 4;
  float d[4][kSqMaxC], rd[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    rd[u] = 0.f;
#pragma unroll
    for (int c = 0; c < kSqMaxC; ++c) d[u][c] = 0.f;
    if (m0 + u < M) {
      const float *dp = dst + ((size_t)b * M + m0 + u) * C;
#pragma unroll
      for (int c = 0; c < kSqMaxC; ++c)
        if (c < C) d[u][c] = dp[c];
      rd[u] = sumsq_cascade(dp, C);
    }
  }
  __syncthreads();
  if (m0 >= M) return;
  const bool vec = (M & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
  const int rows = min(kSqRows, N - n0);
  for (int t = 0; t < rows; ++t) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float zz = __fmul_rn(srow[t][0], d[u][0]);
#pragma unroll
      for (int c = 1; c < kSqMaxC; ++c)
        if (c < C) zz = __fmaf_rn(srow[t][c], d[u][c], zz);
      v[u] = __fadd_rn(__fadd_rn(__fmul_rn(-2.0f, zz), srow[t][kSqMaxC]), rd[u]);
    }
    float *o = out + ((size_t)b * N + n0 + t) * M + m0;
    if (vec) {
      __stcs(reinterpret_cast<float4 *>(o), make_float4(v[0], v[1], v[2], v[3]));
    } else {
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (m0 + u < M) o[u] = v[u];
    }
  }
}

__global__ void __launch_bounds__(256) square_distance_kernel(const float *__restrict__ src,
                                                              const float *__restrict__ dst, int B, int N, int M,
                                                              int C, float *__restrict__ out) {
  const long long total = (long long)B * N * M;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(g % M);
    const long long bn = g / M;
    const int b = (int)(bn / N);
    const float *s = src + (size_t)bn * C;
    const float *d = dst + ((size_t)b * M + m) * C;
    float zz = __fmul_rn(s[0], d[0]);
    for (int c = 1; c < C; ++c) zz = __fmaf_rn(s[c], d[c], zz);
    out[g] = __fadd_rn(__fadd_rn(__fmul_rn(-2.0f, zz), sumsq_cascade(s, C)), sumsq_cascade(d, C));
  }
}

__global__ void __launch_bounds__(128) query_ball_torch_kernel(int N, int S, float radius2, int nsample,
                                                               const float *__restrict__ xyz,
                                                               const float *__restrict__ new_xyz,
                                                               long long *__restrict__ group_idx) {
  const int b = blockIdx.y, lane = threadIdx.x & 31;
  const int s = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (s >= S) return;
  const float *p = xyz + (size_t)b * N * 3;
  const float *q = new_xyz + ((size_t)b * S + s) * 3;
  long long *o = group_idx + ((size_t)b * S + s) * nsample;
  const float q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2);
  const float rs = hg_sumsq3_seq(q0, q1, q2);
  int cnt = 0, first = N;
  for (int k0 = 0; k0 < N && cnt < nsample; k0 += 32) {
    const int k = k0 + lane;
    bool hit = false;
    if (k < N) {
      const float x = __ldg(p + (size_t)k * 3), y = __ldg(p + (size_t)k * 3 + 1), z = __ldg(p + (size_t)k * 3 + 2);
      const float zz = hg_dot3_fma(q0, q1, q2, x, y, z);
      const float d = __fadd_rn(__fadd_rn(__fmul_rn(-2.0f, zz), rs), hg_sumsq3_seq(x, y, z));
      hit = !(d > radius2);
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
  for (int l = cnt + lane; l < nsample; l += 32) o[l] = first;  // empty ball -> N, as the reference's sort leaves it
}

// index_points: out[b,e,:] = points[b, idx[b,e], :]
// Two shapes matter (model/pointnet2_utils.py:110-138 sample_and_group): coordinate rows (C = 3: one thread per row,
// the index read once, 32-bit arithmetic) and feature rows (C a multiple of 4: one 16-byte chunk per thread).  The
// generic kernel does 64-bit divisions per ELEMENT, which cost more than the copy.
template <int C>
__global__ void __launch_bounds__(256) index_points_rows_kernel(const float *__restrict__ points,
                                                                const long long *__restrict__ idx, int N, int M,
                                                                unsigned rows, float *__restrict__ out) {
  for (unsigned r = blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += gridDim.x * blockDim.x) {
    const unsigned b = r / (unsigned)M;
    const float *src = points + ((size_t)b * N + (size_t)idx[r]) * C;
    float v[C];
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = __ldg(src + c);
#pragma unroll
    for (int c = 0; c < C; ++c) out[(size_t)r * C + c] = v[c];
  }
}

__global__ void __launch_bounds__(256) index_points_vec4_kernel(const float *__restrict__ points,
                                                                const long long *__restrict__ idx, int N, int M, int C4,
                                                                unsigned chunks, float4 *__restrict__ out) {
  for (unsigned g = blockIdx.x * blockDim.x + threadIdx.x; g < chunks; g += gridDim.x * blockDim.x) {
    const unsigned r = g / (unsigned)C4, c4 = g - r * (unsigned)C4;
    const unsigned b = r / (unsigned)M;
    out[g] = __ldg(reinterpret_cast<const float4 *>(points + ((size_t)b * N + (size_t)idx[r]) * (4 * (size_t)C4)) + c4);
  }
}

__global__ void __launch_bounds__(256) index_points_kernel(const float *__restrict__ points,
                                                           const long long *__restrict__ idx, int B, int N, int C,
                                                           int M, float *__restrict__ out) {
  const long long total = (long long)B * M * C;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(g % C);
    const long long be = g / C;
    const int b = (int)(be / M);
    const long long a = idx[be];
    out[g] = __ldg(points + ((size_t)b * N + (size_t)a) * C + c);
  }
}

__global__ void idx64_to_keys_kernel(const long long *__restrict__ idx, long long total, int N, int *__restrict__ keys) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long a = idx[g];
    keys[g] = (a >= 0 && a < N) ? (int)a : -1;
  }
}

// grad_points[b,n,:] = sum over edges e with idx[b,e]==n, ascending e, of grad_out[b,e,:]
__global__ void __launch_bounds__(256) index_points_grad_kernel(const float *__restrict__ grad_out,
                                                                const int *__restrict__ off,
                                                                const int *__restrict__ list, int B, int N, int C,
                                                                int M, float *__restrict__ grad_points) {
  const long long total = (long long)B * N * C;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(g % C);
    const long long bn = g / C;
    const int b = (int)(bn / N), n = (int)(bn % N);
    const int *o = off + (size_t)b * (N + 1);
    const int *l = list + (size_t)b * M;
    float acc = 0.f;
    for (int q = o[n]; q < o[n + 1]; ++q) acc = __fadd_rn(acc, grad_out[((size_t)b * M + l[q]) * C + c]);
    grad_points[g] = acc;
  }
}

}  // namespace

HG_API int hg_square_distance_f32(const float *src, const float *dst, int B, int N, int M, int C, float *out,
                                  hgStream stream_) {
  HG_NVTX_RANGE("hg_square_distance_f32");
  HG_REQUIRE(src && dst && out, HG_E_BADARG, "square_distance: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && M > 0 && C > 0, HG_E_BADARG, "square_distance: sizes must be positive");
  if (C <= kSqMaxC && B <= 65535 && (N + kSqRows - 1) / kSqRows <= 65535) {
    dim3 grid((M + 1023) / 1024, (N + kSqRows - 1) / kSqRows, B);
    square_distance_small_c_kernel<<<grid, 256, 0, hg_stream(stream_)>>>(src, dst, N, M, C, out);
  } else {
    const long long total = (long long)B * N * M;
    square_distance_kernel<<<hg_grid_for(total, 256, 32), 256, 0, hg_stream(stream_)>>>(src, dst, B, N, M, C, out);
  }
  HG_CHECK_LAUNCH("square_distance");
  return HG_OK;
}

HG_API int hg_query_ball_torch_f32(float radius2, int nsample, const float *xyz, const float *new_xyz, int B, int N,
                                   int S, int64_t *group_idx, hgStream stream_) {
  HG_NVTX_RANGE("hg_query_ball_torch_f32");
  HG_REQUIRE(xyz && new_xyz && group_idx, HG_E_BADARG, "query_ball_torch: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && S > 0 && nsample > 0, HG_E_BADARG, "query_ball_torch: sizes must be positive");
  HG_REQUIRE(B <= 65535, HG_E_UNSUPPORTED, "query_ball_torch: B=%d > 65535", B);
  query_ball_torch_kernel<<<dim3((S + 3) / 4, B), 128, 0, hg_stream(stream_)>>>(N, S, radius2, nsample, xyz, new_xyz,
                                                                                (long long *)group_idx);
  HG_CHECK_LAUNCH("query_ball_torch");
  return HG_OK;
}

HG_API int hg_index_points_f32(const float *points, const int64_t *idx, int B, int N, int C, int M, float *out,
                               hgStream stream_) {
  HG_NVTX_RANGE("hg_index_points_f32");
  HG_REQUIRE(points && idx && out, HG_E_BADARG, "index_points: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && C > 0 && M > 0, HG_E_BADARG, "index_points: sizes must be positive");
  const long long total = (long long)B * M * C, rows = (long long)B * M;
  const bool aligned = ((reinterpret_cast<uintptr_t>(points) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  if (C == 3 && rows < (1LL << 31)) {
    index_points_rows_kernel<3><<<hg_grid_for(rows, 256, 32), 256, 0, hg_stream(stream_)>>>(points, (const long long *)idx, N, M,
                                                                                           (unsigned)rows, out);
  } else if ((C & 3) == 0 && aligned && total / 4 < (1LL << 31)) {
    index_points_vec4_kernel<<<hg_grid_for(total / 4, 256, 32), 256, 0, hg_stream(stream_)>>>(
        points, (const long long *)idx, N, M, C / 4, (unsigned)(total / 4), reinterpret_cast<float4 *>(out));
  } else {
    index_points_kernel<<<hg_grid_for(total, 256, 32), 256, 0, hg_stream(stream_)>>>(points, (const long long *)idx, B, N, C, M,
                                                                                     out);
  }
  HG_CHECK_LAUNCH("index_points");
  return HG_OK;
}

HG_API size_t hg_index_points_grad_workspace_bytes(int B, int N, int M) {
  if (B <= 0 || N <= 0 || M <= 0) return 0;
  return hg_layout_bytes<HgKeysCsr>(B, N, (long long)M, true);
}

HG_API int hg_index_points_grad_f32(const float *grad_out, const int64_t *idx, int B, int N, int C, int M,
                                    float *grad_points, void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_index_points_grad_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(grad_out && idx && grad_points, HG_E_BADARG, "index_points_grad: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && C > 0 && M > 0, HG_E_BADARG, "index_points_grad: sizes must be positive");
  HG_REQUIRE(workspace && workspace_bytes >= hg_index_points_grad_workspace_bytes(B, N, M), HG_E_WORKSPACE,
             "index_points_grad: workspace too small");
  const auto w = hg_layout_at<HgKeysCsr>(workspace, B, N, (long long)M, true);
  const long long te = (long long)B * M;
  idx64_to_keys_kernel<<<hg_grid_for(te, 256, 32), 256, 0, stream>>>((const long long *)idx, te, N, w.keys);
  HG_CHECK_LAUNCH("idx64_to_keys");
  HgCsr csr;
  int rc = hg_csr_build(w.keys, B, M, N, w.csr.ptr, w.csr.bytes, &csr, stream);
  if (rc) return rc;
  const long long total = (long long)B * N * C;
  index_points_grad_kernel<<<hg_grid_for(total, 256, 32), 256, 0, stream>>>(grad_out, csr.off, csr.list, B, N, C, M,
                                                                            grad_points);
  HG_CHECK_LAUNCH("index_points_grad");
  return HG_OK;
}
