// hg_knn.cu -- k-nearest-neighbour selection and the kNN-outlier loss.
//
//   hg_knn_self_f32         util/dist_utils.py:148-156 (KNNDist) and model/dgcnn_cls.py:8-12 (DGCNN knn)
//   hg_knn_outlier_fwd/bwd  util/dist_utils.py:157-172 and its autograd backward
//   hg_knn_points_f32       pytorch3d.ops.knn_points (third party; semantics restated, see DESIGN.md)
//
// Reference arithmetic (bit-exact restatement, SURVEY.md section 8 a-bis):
//   xx_i = (p0*p0 + p1*p1) + p2*p2           torch.sum(pc**2, dim)   [ATen cascade of 16s for C >= 16]
//   zz   = fma(p_i[C-1],p_j[C-1], ... p_i[0]*p_j[0])                 torch.matmul, sequential FMA chain
//   dist[i,j] = (xx_j + (-2*zz)) + xx_i      (DGCNN's pairwise_distance is exactly -dist)
// Selection: the k1 smallest per row, ascending, lowest index first among equal values (canonical order;
// torch.topk leaves tie order unspecified).  The matrix [B,K,K] is never stored for C == 3 (hg_knn3.cu).
#include "hg_common.cuh"

namespace {

// ---- generic channel count (DGCNN edge-conv layers 2-4: C = 64, 64, 128) ------------------------------------
// xx with ATen's cascade-sum order (levels of 16): probed bit-exact for C = 64, 128.
__global__ void knn_sumsq_kernel(const float *__restrict__ pc, long long total, int C, float *__restrict__ xx) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const float *a = pc + (size_t)g * C;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
    if ((C & 15) == 0 && (reinterpret_cast<uintptr_t>(pc) & 15) == 0) {  // same order, 16-byte loads, 16 channels per step
      for (int c = 0; c < C; c += 16) {
        float4 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldg(reinterpret_cast<const float4 *>(a + c) + u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          acc0 = __fadd_rn(acc0, __fmul_rn(v[u].x, v[u].x));
          acc0 = __fadd_rn(acc0, __fmul_rn(v[u].y, v[u].y));
          acc0 = __fadd_rn(acc0, __fmul_rn(v[u].z, v[u].z));
          acc0 = __fadd_rn(acc0, __fmul_rn(v[u].w, v[u].w));
        }
        acc1 = __fadd_rn(acc1, acc0);
        acc0 = 0.f;
        if (((c + 16) & 255) == 0) {
          acc2 = __fadd_rn(acc2, acc1);
          acc1 = 0.f;
        }
      }
      xx[g] = __fadd_rn(__fadd_rn(acc0, acc1), acc2);
      continue;
    }
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
    xx[g] = __fadd_rn(__fadd_rn(acc0, acc1), acc2);
  }
}

// dist tile: 128 rows x 128 columns per CTA, 8 x 8 per thread (columns as four packed pairs), channels consumed strictly
// in order: every accumulator is the reference's sequential FMA chain (product of channel 0 first, then c = 1..C-1).
// Per channel a thread reads 8 row values (two broadcast LDS.128) and 8 column values (two LDS.128) for 32 FFMA2:
// FMA-bound, where the first version (4 x 4 scalar, 8 LDS.32 per 16 FFMA) was LSU-bound.
constexpr int kGTM = 128, kGTN = 128, kGC = 16;
__global__ void __launch_bounds__(256) knn_dist_generic_kernel(const float *__restrict__ pc,
                                                               const float *__restrict__ xx, int K, int C,
                                                               float *__restrict__ dist /*[nb,K,K]*/) {
  __shared__ __align__(16) float As[kGC][kGTM], Bs[kGC][kGTN];
  const int b = blockIdx.z;
  const float *p = pc + (size_t)b * K * C;
  const int i0 = blockIdx.y * kGTM, j0 = blockIdx.x * kGTN;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float2 acc[8][4];
#pragma unroll
  for (int u = 0; u < 8; ++u) acc[u][0] = acc[u][1] = acc[u][2] = acc[u][3] = make_float2(0.f, 0.f);
  const bool vec_ok = (C & 3) == 0 && (reinterpret_cast<uintptr_t>(pc) & 15) == 0;
  for (int c0 = 0; c0 < C; c0 += kGC) {
    __syncthreads();
    // stage kGC channels of the 128 rows and the 64 columns, transposed to [channel][point]
    for (int t = threadIdx.x; t < (kGTM + kGTN) * (kGC / 4); t += 256) {
      const int pt = t % (kGTM + kGTN), q = t / (kGTM + kGTN);
      const bool isA = pt < kGTM;
      const int row = isA ? i0 + pt : j0 + (pt - kGTM);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const int c = c0 + 4 * q;
      if (row < K) {
        const float *src = p + (size_t)row * C + c;
        if (vec_ok && c + 3 < C) {
          v = *reinterpret_cast<const float4 *>(src);
        } else {
          if (c < C) v.x = src[0];
          if (c + 1 < C) v.y = src[1];
          if (c + 2 < C) v.z = src[2];
          if (c + 3 < C) v.w = src[3];
        }
      }
      float *dstp = isA ? &As[4 * q][pt] : &Bs[4 * q][pt - kGTM];
      const int ld = isA ? kGTM : kGTN;
      dstp[0] = v.x;
      dstp[ld] = v.y;
      dstp[2 * ld] = v.z;
      dstp[3 * ld] = v.w;
    }
    __syncthreads();
    const int cl = min(kGC, C - c0);
#pragma unroll 4
    for (int cc = 0; cc < cl; ++cc) {
      const float4 a0 = *reinterpret_cast<const float4 *>(&As[cc][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4 *>(&As[cc][ty * 8 + 4]);
      const float4 bb = *reinterpret_cast<const float4 *>(&Bs[cc][tx * 4]);       // columns tx*4 .. +3
      const float4 bc = *reinterpret_cast<const float4 *>(&Bs[cc][64 + tx * 4]);  // columns 64 + tx*4 .. +3 (no bank conflicts)
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float2 b01 = make_float2(bb.x, bb.y), b23 = make_float2(bb.z, bb.w), b45 = make_float2(bc.x, bc.y),
                   b67 = make_float2(bc.z, bc.w);
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        acc[u][0] = __ffma2_rn(make_float2(a[u], a[u]), b01, acc[u][0]);
        acc[u][1] = __ffma2_rn(make_float2(a[u], a[u]), b23, acc[u][1]);
        acc[u][2] = __ffma2_rn(make_float2(a[u], a[u]), b45, acc[u][2]);
        acc[u][3] = __ffma2_rn(make_float2(a[u], a[u]), b67, acc[u][3]);
      }
    }
  }
  const float *xb = xx + (size_t)b * K;
  const int j = j0 + tx * 4;  // this thread's columns: j .. j+3 and j+64 .. j+67
  float xj[8];
#pragma unroll
  for (int v = 0; v < 8; ++v) {
    const int jj = j + (v & 3) + ((v >> 2) << 6);
    xj[v] = (jj < K) ? xb[jj] : 0.f;
  }
  const bool vst = (K & 3) == 0 && (reinterpret_cast<uintptr_t>(dist) & 15) == 0;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const int i = i0 + ty * 8 + u;
    if (i >= K) continue;
    const float xi = xb[i];
    float o[8];
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      o[2 * v] = __fadd_rn(__fadd_rn(xj[2 * v], __fmul_rn(-2.0f, acc[u][v].x)), xi);
      o[2 * v + 1] = __fadd_rn(__fadd_rn(xj[2 * v + 1], __fmul_rn(-2.0f, acc[u][v].y)), xi);
    }
    float *dp = dist + ((size_t)b * K + i) * K + j;
    if (vst && j + 3 < K) {
      *reinterpret_cast<float4 *>(dp) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
      for (int v = 0; v < 4; ++v)
        if (j + v < K) dp[v] = o[v];
    }
    if (vst && j + 67 < K) {
      *reinterpret_cast<float4 *>(dp + 64) = make_float4(o[4], o[5], o[6], o[7]);
    } else {
#pragma unroll
      for (int v = 0; v < 4; ++v)
        if (j + 64 + v < K) dp[64 + v] = o[4 + v];
    }
  }
}

// Warp per row.  The k1 smallest (value, index) pairs of a row of K distances, ascending, lowest index first on ties.
//   1. every lane takes the minimum of its K/32 strided elements; the k1-th smallest of those 32 lane minima (one
//      warp-wide bitonic sort) is an upper bound tau on the row's k1-th smallest value (k1 <= 32 distinct elements
//      are <= tau);
//   2. the elements <= tau -- typically 1.5-2 k1 of them -- are compacted in index order into a small candidate
//      buffer (ballot + prefix popcount);
//   3. k1 rounds of "smallest (value, index) strictly after the previous pick" run over the candidates only.
// The first version ran step 3 over the whole row (k1 x K/32 steps per lane).  If the candidates overflow the buffer
// (heavy ties), the row falls back to exactly that.
// Long lists (kLong: 33 <= k1 <= 64) bound with the TWO smallest strided elements of every lane instead: the k1-th
// smallest of those 64 distinct elements (one 64-wide bitonic sort, two per lane) is again an upper bound, and the
// candidate buffer is twice as large.
constexpr int kSelCap = 128;      // candidates per row kept in shared memory (4 per lane)
constexpr int kSelCapLong = 256;  // the same for long lists (8 per lane)
__host__ __device__ constexpr int knn_sel_cap(bool long_list) { return long_list ? kSelCapLong : kSelCap; }

__device__ __forceinline__ void knn_select_rounds(const float *__restrict__ v, const int *__restrict__ id, int n,
                                                  int k1, int lane, float *__restrict__ vals, int *__restrict__ idx,
                                                  size_t out) {
  float pv = -CUDART_INF_F;
  int pj = -1;
  for (int t = 0; t < k1; ++t) {
    float bv = CUDART_INF_F;
    int bj = 0x7fffffff;
    for (int q = lane; q < n; q += 32) {
      const float x = v[q];
      const int j = id ? id[q] : q;
      const bool after = (x > pv) || (x == pv && j > pj);
      if (after && (x < bv || (x == bv && j < bj))) {
        bv = x;
        bj = j;
      }
    }
    const float wv = hg_warp_min_f32(bv);
    const int wj = __reduce_min_sync(0xffffffffu, (bv == wv) ? bj : 0x7fffffff);
    pv = wv;
    pj = wj;
    if (lane == 0) {
      if (vals) vals[out + t] = wv;
      idx[out + t] = wj;
    }
  }
}

template <bool kLong>
__global__ void __launch_bounds__(128) knn_select_rows_kernel(const float *__restrict__ dist, int nrows, int K,
                                                              int k1, float *__restrict__ vals,
                                                              int *__restrict__ idx) {
  constexpr int kCap = knn_sel_cap(kLong);
  extern __shared__ float rowbuf[];  // [4 warps][K] rows, then [4][kCap] candidate values, [4][kCap] indices
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *row = rowbuf + (size_t)warp * K;
  float *cv = rowbuf + (size_t)4 * K + (size_t)warp * kCap;
  int *ci = reinterpret_cast<int *>(rowbuf + (size_t)4 * K + (size_t)4 * kCap) + (size_t)warp * kCap;
  for (int r = blockIdx.x * 4 + warp; r < nrows; r += gridDim.x * 4) {
    __syncwarp();
    float lmin = CUDART_INF_F, lmin2 = CUDART_INF_F;  // (lmin2: the second smallest, long lists only)
    for (int j = lane; j < K; j += 32) {
      const float x = dist[(size_t)r * K + j];
      row[j] = x;
      if (kLong) {  // (a NaN compares false and is skipped, as fminf skips it)
        if (x < lmin) {
          lmin2 = lmin;
          lmin = x;
        } else if (x < lmin2) {
          lmin2 = x;
        }
      } else {
        lmin = fminf(lmin, x);
      }
    }
    float tau;
    if (kLong) {
      // bitonic sort of the 64 values (element e = lane + 32 r held as s[r]), ascending; stride 32 pairs a lane's own
      // two values, and the size-32 blocks run ascending for r = 0, descending for r = 1
      float s[2] = {lmin, lmin2};
#pragma unroll
      for (int size = 2; size <= 64; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
          if (stride == 32) {
            const float lo = fminf(s[0], s[1]), hi = fmaxf(s[0], s[1]);
            s[0] = lo;
            s[1] = hi;
            continue;
          }
          const bool lower = ((lane & stride) == 0);
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float o = __shfl_xor_sync(0xffffffffu, s[h], stride);
            const bool up = size == 64 ? true : size == 32 ? h == 0 : ((lane & size) == 0);
            s[h] = (up == lower) ? fminf(s[h], o) : fmaxf(s[h], o);
          }
        }
      }
      tau = __shfl_sync(0xffffffffu, s[1], k1 - 33);  // element k1 - 1 >= 32
    } else {
      // bitonic sort of the 32 lane minima across the warp (ascending by lane)
      float s = lmin;
#pragma unroll
      for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
          const float o = __shfl_xor_sync(0xffffffffu, s, stride);
          const bool up = ((lane & size) == 0);         // ascending block
          const bool lower = ((lane & stride) == 0);    // this lane keeps the smaller of the pair in an ascending block
          s = (up == lower) ? fminf(s, o) : fmaxf(s, o);
        }
      }
      tau = __shfl_sync(0xffffffffu, s, k1 - 1);
    }
    __syncwarp();
    int cnt = 0;
    for (int j0 = 0; j0 < K; j0 += 32) {
      const int j = j0 + lane;
      const float x = (j < K) ? row[j] : CUDART_INF_F;
      const bool keep = (j < K) && (x <= tau);
      const unsigned m = __ballot_sync(0xffffffffu, keep);
      const int pos = cnt + __popc(m & ((1u << lane) - 1u));
      if (keep && pos < kCap) {
        cv[pos] = x;
        ci[pos] = j;
      }
      cnt += __popc(m);
    }
    __syncwarp();
    if (cnt <= kCap)
      knn_select_rounds(cv, ci, cnt, k1, lane, vals, idx, (size_t)r * k1);
    else
      knn_select_rounds(row, nullptr, K, k1, lane, vals, idx, (size_t)r * k1);
  }
}

// ---- kNN-outlier loss ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) knn_outlier_fwd_kernel(const float *__restrict__ vals, int K, int k1,
                                                              float alpha, const float *__restrict__ weights,
                                                              float *__restrict__ value, float *__restrict__ mask,
                                                              float *__restrict__ loss) {
  const int b = blockIdx.x, tid = threadIdx.x;
  __shared__ double red[256];
  __shared__ float thr_s;
  const float *v = vals + (size_t)b * K * k1;
  float *val = value + (size_t)b * K;
  const float kf = (float)(k1 - 1);
  double s = 0.0;
  for (int i = tid; i < K; i += 256) {
    float acc = v[(size_t)i * k1 + 1];
    for (int t = 2; t < k1; ++t) acc = __fadd_rn(acc, v[(size_t)i * k1 + t]);
    const float x = __fdiv_rn(acc, kf);
    val[i] = x;
    s += (double)x;
  }
  red[tid] = s;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (tid < st) red[tid] += red[tid + st];
    __syncthreads();
  }
  const double mean = red[0] / (double)K;
  __syncthreads();
  double ss = 0.0;
  for (int i = tid; i < K; i += 256) {
    const double d = (double)val[i] - mean;
    ss += d * d;
  }
  red[tid] = ss;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (tid < st) red[tid] += red[tid + st];
    __syncthreads();
  }
  if (tid == 0) {
    const float stdf = (float)sqrt(red[0] / (double)(K - 1));  // torch.std: unbiased
    thr_s = __fadd_rn((float)mean, __fmul_rn(alpha, stdf));
  }
  __syncthreads();
  const float thr = thr_s;
  double l = 0.0;
  for (int i = tid; i < K; i += 256) {
    const float m = val[i] > thr ? 1.f : 0.f;
    mask[(size_t)b * K + i] = m;
    l += (double)__fmul_rn(val[i], m);
  }
  __syncthreads();
  red[tid] = l;
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (tid < st) red[tid] += red[tid + st];
    __syncthreads();
  }
  if (tid == 0) {
    const float lb = (float)(red[0] / (double)K);
    loss[b] = weights ? __fmul_rn(lb, weights[b]) : lb;
  }
}

__global__ void knn_bwd_keys_kernel(const int *__restrict__ idx, const float *__restrict__ mask, long long total,
                                    int k1, int *__restrict__ keys) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(g % k1);
    const long long row = g / k1;
    keys[g] = (t >= 1 && mask[row] != 0.f) ? idx[g] : -1;
  }
}

// grad[n] = coef * ( [mask_n] sum_t 2(p_n - p_{idx[n,t]})  +  sum_{edges (i,t)->n, mask_i} 2(p_n - p_i) )
__global__ void __launch_bounds__(256) knn_outlier_bwd_kernel(const float *__restrict__ pc,
                                                              const int *__restrict__ idx,
                                                              const float *__restrict__ mask,
                                                              const float *__restrict__ g, const int *__restrict__ off,
                                                              const int *__restrict__ list,
                                                              const int *__restrict__ keys /*[B,K*k1] edge -> point or -1*/,
                                                              int B, int K, int C, int k1, float *__restrict__ grad) {
  const long long total = (long long)B * K;
  for (long long gi = (long long)blockIdx.x * blockDim.x + threadIdx.x; gi < total;
       gi += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(gi / K), n = (int)(gi % K);
    const float *p = pc + (size_t)b * K * C;
    const float coef = g[b] / ((float)K * (float)(k1 - 1));
    const bool own = mask[gi] != 0.f;
    const int *nb = idx + (size_t)gi * k1;
    const int *o = off + (size_t)b * (K + 1);
    const int *l = list + (size_t)b * K * k1;
    const int p0 = o[n], p1 = o[n + 1];
    if (C == 3) {  // the hot case: walk the neighbour list and the reverse map ONCE for the three coordinates
      const float v0 = p[(size_t)n * 3], v1 = p[(size_t)n * 3 + 1], v2 = p[(size_t)n * 3 + 2];
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
      if (own)
        for (int t = 1; t < k1; ++t) {
          const float *r = p + (size_t)nb[t] * 3;
          a0 += 2.0f * (v0 - r[0]);
          a1 += 2.0f * (v1 - r[1]);
          a2 += 2.0f * (v2 - r[2]);
        }
      if (p1 - p0 <= 32) {
        int e = -1;
        for (int q = p0; q < p1; ++q) {  // ascending edge order, whatever order the list was filled in
          e = hg_csr_next(l, p0, p1, e);
          const float *r = p + (size_t)(e / k1) * 3;
          a0 += 2.0f * (v0 - r[0]);
          a1 += 2.0f * (v1 - r[1]);
          a2 += 2.0f * (v2 - r[2]);
        }
      } else {  // a hub (duplicated points): O(edges) scan of the forward map instead of the O(deg^2) selection walk
        const int *kk = keys + (size_t)b * K * k1;
        for (int e = 0; e < K * k1; ++e)
          if (kk[e] == n) {
            const float *r = p + (size_t)(e / k1) * 3;
            a0 += 2.0f * (v0 - r[0]);
            a1 += 2.0f * (v1 - r[1]);
            a2 += 2.0f * (v2 - r[2]);
          }
      }
      grad[(size_t)gi * 3] = coef * a0;
      grad[(size_t)gi * 3 + 1] = coef * a1;
      grad[(size_t)gi * 3 + 2] = coef * a2;
      continue;
    }
    for (int c = 0; c < C; ++c) {
      const float v = p[(size_t)n * C + c];
      float acc = 0.f;
      if (own)
        for (int t = 1; t < k1; ++t) acc += 2.0f * (v - p[(size_t)nb[t] * C + c]);
      if (p1 - p0 <= 32) {
        int e = -1;
        for (int q = p0; q < p1; ++q) {  // ascending edge order, whatever order the list was filled in
          e = hg_csr_next(l, p0, p1, e);
          acc += 2.0f * (v - p[(size_t)(e / k1) * C + c]);
        }
      } else {
        const int *kk = keys + (size_t)b * K * k1;
        for (int e = 0; e < K * k1; ++e)
          if (kk[e] == n) acc += 2.0f * (v - p[(size_t)(e / k1) * C + c]);
      }
      grad[(size_t)gi * C + c] = coef * acc;
    }
  }
}

// Small 3-D clouds: the whole backward of one cloud in ONE CTA -- keys, reverse map (integer shared-memory atomics:
// counts and slots are order-independent, the walk below is in ascending edge order whatever the slots) and the
// gradient -- instead of keys + memset + count + scan + fill + gradient kernels (53 us of a 385 us config-1 step).
// Same sums in the same order as knn_outlier_bwd_kernel.
constexpr int kBwdSmallSmemMax = 100 * 1024;
__host__ __device__ inline size_t knn_bwd_small_smem(int K, int k1) {
  return ((size_t)K * 3 + (size_t)K + (size_t)(K + 1) + (size_t)K + (size_t)K * (k1 - 1)) * 4;
}

__global__ void __launch_bounds__(256) knn_outlier_bwd_small_kernel(const float *__restrict__ pc,
                                                                    const int *__restrict__ idx,
                                                                    const float *__restrict__ mask,
                                                                    const float *__restrict__ g, int K, int k1,
                                                                    float *__restrict__ grad) {
  extern __shared__ int bsm[];
  float *sp = (float *)bsm;              // [K*3]
  float *smask = sp + (size_t)K * 3;     // [K]
  int *soff = (int *)(smask + K);        // [K+1]
  int *scur = soff + K + 1;              // [K]
  int *slist = scur + K;                 // [<= K*(k1-1)]
  __shared__ int warp_tot[8];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *p = pc + (size_t)b * K * 3;
  const int *ix = idx + (size_t)b * K * k1;
  for (int q = tid; q < K * 3; q += 256) sp[q] = p[q];
  for (int q = tid; q < K; q += 256) smask[q] = mask[(size_t)b * K + q];
  for (int q = tid; q <= K; q += 256) soff[q] = 0;
  __syncthreads();
  // edges leave outlier rows only (mask != 0, a few per cent of the cloud): walk rows, not edges
  auto key_at = [&](int i, int t) -> int {
    const int key = ix[(size_t)i * k1 + t];
    return (key >= 0 && key < K) ? key : -1;
  };
  for (int i = tid; i < K; i += 256)
    if (smask[i] != 0.f)
      for (int t = 1; t < k1; ++t) {
        const int key = key_at(i, t);
        if (key >= 0) atomicAdd(soff + key + 1, 1);
      }
  __syncthreads();
  {  // exclusive scan of the counts: contiguous chunk per thread, warp scan, block carry
    const int per = (K + 255) / 256;
    const int lo = min(tid * per, K), hi = min(lo + per, K);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += soff[i + 1];
    int v = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, v, d);
      if (lane >= d) v += t;
    }
    if (lane == 31) warp_tot[warp] = v;
    __syncthreads();
    int run = v - sum;
    for (int w = 0; w < warp; ++w) run += warp_tot[w];
    for (int i = lo; i < hi; ++i) {
      const int c = soff[i + 1];
      scur[i] = run;
      run += c;
      soff[i + 1] = run;  // (soff[0] stays 0)
    }
  }
  __syncthreads();
  for (int i = tid; i < K; i += 256)
    if (smask[i] != 0.f)
      for (int t = 1; t < k1; ++t) {
        const int key = key_at(i, t);
        if (key >= 0) slist[atomicAdd(scur + key, 1)] = i * k1 + t;
      }
  __syncthreads();
  const float coef = g[b] / ((float)K * (float)(k1 - 1));
  for (int n = tid; n < K; n += 256) {
    const float v0 = sp[n * 3], v1 = sp[n * 3 + 1], v2 = sp[n * 3 + 2];
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    if (smask[n] != 0.f) {
      const int *nb = ix + (size_t)n * k1;
      for (int t = 1; t < k1; ++t) {
        const float *r = sp + (size_t)nb[t] * 3;
        a0 += 2.0f * (v0 - r[0]);
        a1 += 2.0f * (v1 - r[1]);
        a2 += 2.0f * (v2 - r[2]);
      }
    }
    const int p0 = soff[n], p1 = soff[n + 1];
    if (p1 - p0 <= 32) {
      int e = -1;
      for (int q = p0; q < p1; ++q) {
        e = hg_csr_next(slist, p0, p1, e);
        const float *r = sp + (size_t)(e / k1) * 3;
        a0 += 2.0f * (v0 - r[0]);
        a1 += 2.0f * (v1 - r[1]);
        a2 += 2.0f * (v2 - r[2]);
      }
    } else {  // a hub: scan the forward map (ascending edge order = rows, then slots)
      for (int i = 0; i < K; ++i) {
        if (smask[i] == 0.f) continue;
        for (int t = 1; t < k1; ++t)
          if (key_at(i, t) == n) {
            const float *r = sp + (size_t)i * 3;
            a0 += 2.0f * (v0 - r[0]);
            a1 += 2.0f * (v1 - r[1]);
            a2 += 2.0f * (v2 - r[2]);
          }
      }
    }
    float *go = grad + ((size_t)b * K + n) * 3;
    go[0] = coef * a0;
    go[1] = coef * a1;
    go[2] = coef * a2;
  }
}

constexpr size_t kGenericScratchBytes = (size_t)256 << 20;

// feature clouds: squared norms [B,K], then distance matrices for nb clouds (as many as kGenericScratchBytes holds, >= 1)
struct KnnGenericWorkspace {
  int nb;
  float *xx, *dist;
  KnnGenericWorkspace(HgCarve &c, int B, int K) {
    const size_t per = (size_t)K * K, fit = kGenericScratchBytes / (per * sizeof(float));
    nb = fit < 1 ? 1 : fit > (size_t)B ? B : (int)fit;
    xx = c.take<float>((size_t)B * K), dist = c.take<float>(nb * per);
  }
};

}  // namespace

HG_API size_t hg_knn_self_workspace_bytes(int B, int K, int C, int k1) {
  if (B <= 0 || K <= 0 || C <= 0) return 0;
  return C == 3 ? hg_knn3_self_workspace_bytes(B, K, k1) : hg_layout_bytes<KnnGenericWorkspace>(B, K);
}

HG_API int hg_knn_self_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx, void *workspace,
                           size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_self_f32");
  return hg_knn_self_temporal_f32(pc, B, K, C, k1, vals, idx, nullptr, 0, workspace, workspace_bytes, stream_);
}

HG_API int hg_knn_self_temporal_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx, int *idx_state,
                                    int state_valid, void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_self_temporal_f32");
  return hg_knn_self_temporal_order_f32(pc, B, K, C, k1, vals, idx, idx_state, state_valid, nullptr, workspace,
                                        workspace_bytes, stream_);
}

HG_API int hg_knn_self_temporal_order_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx,
                                          int *idx_state, int state_valid, void *order, void *workspace,
                                          size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_self_temporal_order_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(pc && idx, HG_E_BADARG, "knn_self: null pointer");
  HG_REQUIRE(((uintptr_t)order & 15) == 0, HG_E_BADARG, "knn_self: the ordering state must be 16-byte aligned");
  HG_REQUIRE(B > 0 && K > 0 && C > 0, HG_E_BADARG, "knn_self: sizes must be positive");
  HG_REQUIRE(k1 >= 1 && k1 <= 64 && k1 <= K, HG_E_BADARG, "knn_self: need 1 <= k <= min(64, K); got k=%d K=%d", k1, K);
  HG_REQUIRE(B <= 65535, HG_E_UNSUPPORTED, "knn_self: B=%d > 65535 clouds per call", B);
  if (C == 3)
    return hg_knn3_self_i32(pc, B, K, k1, vals, idx, idx_state, state_valid, order, workspace, workspace_bytes, stream);
  const size_t need = hg_knn_self_workspace_bytes(B, K, C, k1);
  HG_REQUIRE(workspace && workspace_bytes >= need, HG_E_WORKSPACE, "knn_self: workspace too small (%zu < %zu)",
             workspace_bytes, need);
  // the FP32 row select stages four rows of K distances per CTA; beyond that only the tensor-core kernel runs
  const bool rows_fit = (size_t)K * sizeof(float) * 4 <= 200 * 1024;
  const bool tc_shape = hg_knn_tc_supported_feature(K, C, k1) && (reinterpret_cast<uintptr_t>(pc) & 15) == 0;
  HG_REQUIRE(rows_fit || tc_shape, HG_E_UNSUPPORTED, "knn_self: K=%d too large for C=%d path", K, C);
  HG_REQUIRE(rows_fit || g_hg_tune_knn_tc_off != 1, HG_E_UNSUPPORTED,
             "knn_self: hg_tune(\"knn_tc\", 1) selects the FP32 path, which takes K <= 12800 (got K=%d)", K);
  const auto [nb, xx, dist] = hg_layout_at<KnnGenericWorkspace>(workspace, B, K);
  knn_sumsq_kernel<<<hg_grid_for((long long)B * K, 256, 16), 256, 0, stream>>>(pc, (long long)B * K, C, xx);
  HG_CHECK_LAUNCH("knn_sumsq_kernel");
  // feature clouds of DGCNN's shapes: tensor-core filter fused with the exact FP32 evaluation (hg_knn_tc.cu); everything
  // else (and hg_tune("knn_tc", 1)) takes the FP32 distance tile + row select below
  // (small batches leave the serial chain of a CTA exposed -- measured at K = 1024, C = 64: 16 clouds 85 us against
  // 143 us, 8 clouds 82 against 95, 4 clouds 79 against 65 -- so fewer CTAs than a quarter of the SMs stay on the FP32
  // path unless hg_tune("knn_tc", 2) forces the tensor-core kernel; long lists, k1 > 32, need half the SMs -- measured at
  // 2048 x 64, k = 40: 4 clouds 143 us FP32 against 153 tensor-core, 8 clouds 283 against 157, 32 clouds 1121 against 393).
  // Past 4096 points the batch rule does not apply: each CTA walks 17..64 tiles, and the tensor-core kernel won at every
  // batch measured, from one cloud up (8192 x 64, k = 40: 362 us against 952 at one cloud, 907 against 7534 at eight;
  // DESIGN.md section 5.2).  Past 12800 points it is the only route.
  const long long tc_ctas = (long long)B * ((K + 127) / 128);
  const bool tc_fills = (k1 > 32 ? 2 : 4) * tc_ctas >= hg_sm_count() || g_hg_tune_knn_tc_off == 2 || g_hg_tune_knn_tc_off == 5;
  if (g_hg_tune_knn_tc_off != 1 && tc_shape && (tc_fills || K > 4096))
    return hg_knn_tc_run(pc, xx, B, K, C, k1, vals, idx, stream);
  const bool long_list = k1 > 32;
  const size_t sel_smem = ((size_t)4 * K + (size_t)8 * knn_sel_cap(long_list)) * sizeof(float);
  if (sel_smem > 48 * 1024)
    HG_CUDA(cudaFuncSetAttribute(long_list ? knn_select_rows_kernel<true> : knn_select_rows_kernel<false>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
  for (int b0 = 0; b0 < B; b0 += nb) {
    const int cb = (B - b0 < nb) ? (B - b0) : nb;
    dim3 grid((K + kGTN - 1) / kGTN, (K + kGTM - 1) / kGTM, cb);
    knn_dist_generic_kernel<<<grid, 256, 0, stream>>>(pc + (size_t)b0 * K * C, xx + (size_t)b0 * K, K, C, dist);
    HG_CHECK_LAUNCH("knn_dist_generic_kernel");
    const int nrows = cb * K;
    (long_list ? knn_select_rows_kernel<true> : knn_select_rows_kernel<false>)<<<hg_grid_for((long long)nrows * 32, 128, 16),
                                                                                 128, sel_smem, stream>>>(
        dist, nrows, K, k1, vals ? vals + (size_t)b0 * K * k1 : nullptr, idx + (size_t)b0 * K * k1);
    HG_CHECK_LAUNCH("knn_select_rows_kernel");
  }
  return HG_OK;
}

HG_API int hg_knn_points_f32(const float *p1, const float *p2, int B, int N, int M, int K, float *dists, int64_t *idx,
                             hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_points_f32");
  HG_REQUIRE(p1 && p2 && idx, HG_E_BADARG, "knn_points: null pointer");
  HG_REQUIRE(B > 0 && N > 0 && M > 0, HG_E_BADARG, "knn_points: sizes must be positive");
  HG_REQUIRE(K >= 1 && K <= 64 && K <= M, HG_E_BADARG, "knn_points: need 1 <= K <= min(64, M); got K=%d M=%d", K, M);
  HG_REQUIRE(B <= 65535, HG_E_UNSUPPORTED, "knn_points: B=%d > 65535 clouds per call", B);
  return hg_knn3_points_i64(p1, p2, B, N, M, K, dists, (long long *)idx, hg_stream(stream_));
}

HG_API int hg_knn_outlier_fwd_f32(const float *vals, int B, int K, int k1, float alpha, const float *weights,
                                  float *value, float *mask, float *loss, hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_outlier_fwd_f32");
  HG_REQUIRE(vals && value && mask && loss, HG_E_BADARG, "knn_outlier_fwd: null pointer");
  HG_REQUIRE(B > 0 && K > 1 && k1 >= 2, HG_E_BADARG, "knn_outlier_fwd: need K > 1 and k >= 1");
  knn_outlier_fwd_kernel<<<B, 256, 0, hg_stream(stream_)>>>(vals, K, k1, alpha, weights, value, mask, loss);
  HG_CHECK_LAUNCH("knn_outlier_fwd_kernel");
  return HG_OK;
}

HG_API size_t hg_knn_outlier_bwd_workspace_bytes(int B, int K, int k1) {
  if (B <= 0 || K <= 0 || k1 <= 0) return 0;
  return hg_layout_bytes<HgKeysCsr>(B, K, (long long)K * k1, false);
}

HG_API int hg_knn_outlier_bwd_f32(const float *pc, const int *idx, const float *mask, const float *g, int B, int K,
                                  int C, int k1, float *grad_pc, void *workspace, size_t workspace_bytes,
                                  hgStream stream_) {
  HG_NVTX_RANGE("hg_knn_outlier_bwd_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(pc && idx && mask && g && grad_pc, HG_E_BADARG, "knn_outlier_bwd: null pointer");
  HG_REQUIRE(B > 0 && K > 1 && C > 0 && k1 >= 2, HG_E_BADARG, "knn_outlier_bwd: bad sizes");
  HG_REQUIRE(workspace && workspace_bytes >= hg_knn_outlier_bwd_workspace_bytes(B, K, k1), HG_E_WORKSPACE,
             "knn_outlier_bwd: workspace too small");
  if (C == 3 && knn_bwd_small_smem(K, k1) <= (size_t)kBwdSmallSmemMax && !g_hg_tune_small_fused_off) {
    static HgPerDeviceOnce once;
    if (once.first())
      HG_CUDA(cudaFuncSetAttribute(knn_outlier_bwd_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   kBwdSmallSmemMax));
    knn_outlier_bwd_small_kernel<<<B, 256, knn_bwd_small_smem(K, k1), stream>>>(pc, idx, mask, g, K, k1, grad_pc);
    HG_CHECK_LAUNCH("knn_outlier_bwd_small_kernel");
    return HG_OK;
  }
  const auto w = hg_layout_at<HgKeysCsr>(workspace, B, K, (long long)K * k1, false);
  const long long total = (long long)B * K * k1;
  knn_bwd_keys_kernel<<<hg_grid_for(total, 256, 16), 256, 0, stream>>>(idx, mask, total, k1, w.keys);
  HG_CHECK_LAUNCH("knn_bwd_keys_kernel");
  HgCsr csr;
  int rc = hg_csr_build_unordered(w.keys, B, K * k1, K, w.csr.ptr, w.csr.bytes, &csr, stream);
  if (rc) return rc;
  knn_outlier_bwd_kernel<<<hg_grid_for((long long)B * K, 256, 16), 256, 0, stream>>>(pc, idx, mask, g, csr.off, csr.list, w.keys,
                                                                                     B, K, C, k1, grad_pc);
  HG_CHECK_LAUNCH("knn_outlier_bwd_kernel");
  return HG_OK;
}
