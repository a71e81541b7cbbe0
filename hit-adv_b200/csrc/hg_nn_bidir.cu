// hg_nn_bidir.cu -- fused pairwise-distance + bidirectional nearest neighbour for Chamfer / Hausdorff.
//
// Replaces util/set_distance.py:15-32 (_Distance.batch_pairwise_dist: three torch.bmm that materialise
// xx, yy, zz and P, each [B,N2,N1]) together with the two torch.min reductions of :45-48 / :65-68.
// Nothing of size N2 x N1 is ever stored: HBM traffic is the two clouds in and (min,argmin) out.
//
// Arithmetic (bit-exact restatement of the reference's FP32 matrix, SURVEY.md section 8 a-bis):
//     rx_i = fma(x2,x2, fma(x1,x1, x0*x0))         diag(bmm(x,x^T))
//     zz   = fma(x2,y2, fma(x1,y1, x0*y0))         bmm(x,y^T)
//     P    = (rx_i + ry_j) - 2*zz
// computed as  P = (rx_i + ry_j) + zz',  zz' = fma(x2',y2, fma(x1',y1, x0'*y0)),  x' = -2x  (scaling by -2
// commutes with every rounding, so zz' == -2*zz exactly).
//
// Kernel design for sm_100a.  The inner dimension is 3, so this is FP32-pipe work, not tensor-core work.
// Per pair the FMA pipe must execute 5 operations (FMUL, 2 FFMA, 2 FADD); they are issued as packed
// FMUL2/FFMA2/FADD2 (two ROWS per instruction, the column operand broadcast by the .F32 operand form), which
// halves the issue slots and leaves room for the min bookkeeping on the ALU pipe:
//   * a lane keeps T columns (preds) resident in registers (as scalars) and streams the rows (gts) of the CTA's
//     row block from shared memory, two rows per packed instruction (broadcast LDS.128: row pairs interleaved);
//   * column direction (min over rows): FMNMX3 over two rows at a time into T running minima; which block
//     of kColBatch rows produced the minimum is tracked every kColBatch rows;
//   * row direction (min over columns): FMNMX3 tree over the lane's T values, one CREDUX.MIN.F32 across the
//     warp, and a ballot that records WHICH lane attained it;
//   * only minima are tracked in the loop ("two-level argmin"): the exact first index is recovered by the
//     finish kernel, which re-evaluates the kColBatch rows / T columns named by the coarse id with the same
//     arithmetic and takes the first exact match -- torch.min's first-index tie rule.
// Partial results of different CTAs are merged with 64-bit integer atomicMin on (ordered value bits, coarse
// id): order-independent, hence deterministic.
#include "hg_common.cuh"

namespace {

constexpr int kCsrWalkMax = 32;  // in-degree up to which the backward walks a reverse-map segment by selection
constexpr int kColBatch = 32;  // rows per column-direction tracking batch (and rescan width of the finish kernel)
constexpr int kFinishSmallSmemMax = 100 * 1024;  // both clouds of a pair in shared memory: the small finish kernel

struct NnParams {
  const float *gts;    // [B,N2,3]
  const float *preds;  // [B,N1,3]
  int N2, N1;
  int RB;                       // rows per CTA (multiple of kColBatch)
  unsigned long long *colres;   // [B,N1]  (ord(min over rows) << 32) | global row batch
  unsigned long long *rowres;   // [B,N2]  (ord(min over cols) << 32) | (column group << 5 | lane)
  // null, or the per-cloud info of the two pruned-path orderings: only the clouds they flag are computed here
  const float4 *only_a, *only_b;
};

__device__ __forceinline__ bool nn_skip(const NnParams &p, int b) {
  return p.only_a != nullptr && p.only_a[b].y == 0.f && p.only_b[b].y == 0.f;
}

// exact P for the finish kernel; identical operation sequence to the packed main loop
__device__ __forceinline__ float nn_p_exact(float x0, float x1, float x2, float y0, float y1, float y2) {
  const float rx = hg_dot3_fma(x0, x1, x2, x0, x1, x2);
  const float ry = hg_dot3_fma(y0, y1, y2, y0, y1, y2);
  const float t = __fmaf_rn(-2.0f * x2, y2, __fmaf_rn(-2.0f * x1, y1, __fmul_rn(-2.0f * x0, y0)));
  return __fadd_rn(__fadd_rn(rx, ry), t);
}

// launch bounds: T=16 -> 12 warps per SM (3 per scheduler, <= 170 registers); T=8 -> 16 warps per SM (<= 128)
template <int T, int WARPS>
__global__ void __launch_bounds__(WARPS * 32, (T == 8 ? 16 : 12) / WARPS) nn_bidir_d3_kernel(NnParams p) {
  extern __shared__ float4 smem[];
  // row block, two float4 per ROW PAIR (a,b): A = (xa0',xb0',xa1',xb1'), B = (xa2',xb2',rxa,rxb), x' = -2x;
  // +4 entries so that the software prefetch of the last iteration stays in bounds
  float4 *xs = smem;
  uint4 *rowpart = reinterpret_cast<uint4 *>(smem + p.RB + 4);  // [WARPS][RB/2] (m_a,mask_a,m_b,mask_b)
  // column-direction tracking state, one bank column per thread: running minimum at the last batch boundary and
  // the batch that last lowered it (kept out of the register file: 2*T words per thread)
  float *sprev = reinterpret_cast<float *>(rowpart + (size_t)WARPS * (p.RB / 2));  // [T][WARPS*32]
  int *scid = reinterpret_cast<int *>(sprev + T * WARPS * 32);                     // [T][WARPS*32]

  const int b = blockIdx.z;
  if (nn_skip(p, b)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cgroup = blockIdx.y * WARPS + warp;  // global column group (32*T columns)
  const int cbase = cgroup * 32 * T + lane * T;
  const int r0 = blockIdx.x * p.RB;
  const bool warp_active = cgroup * 32 * T < p.N1;

  // ---- stage the row block; rows past N2 get rx=+inf so they never win a minimum ---------------------------
  const float *gx = p.gts + (size_t)b * p.N2 * 3;
  for (int rp = threadIdx.x; rp < p.RB / 2 + 2; rp += WARPS * 32) {
    float v[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int i = r0 + 2 * rp + h;
      v[h][0] = v[h][1] = v[h][2] = 0.f;
      v[h][3] = CUDART_INF_F;
      if (i < p.N2 && 2 * rp + h < p.RB) {
        const float x0 = __ldg(gx + (size_t)i * 3), x1 = __ldg(gx + (size_t)i * 3 + 1), x2 = __ldg(gx + (size_t)i * 3 + 2);
        v[h][0] = -2.0f * x0;
        v[h][1] = -2.0f * x1;
        v[h][2] = -2.0f * x2;
        v[h][3] = hg_dot3_fma(x0, x1, x2, x0, x1, x2);
      }
    }
    xs[2 * rp] = make_float4(v[0][0], v[1][0], v[0][1], v[1][1]);
    xs[2 * rp + 1] = make_float4(v[0][2], v[1][2], v[0][3], v[1][3]);
  }

  // ---- this lane's T columns as scalars; columns past N1 get ry=+inf ----------------------------------------
  float y0[T], y1[T], y2[T], ry[T];
  const float *gy = p.preds + (size_t)b * p.N1 * 3;
#pragma unroll
  for (int t = 0; t < T; ++t) {
    const int j = cbase + t;
    y0[t] = y1[t] = y2[t] = 0.f;
    ry[t] = CUDART_INF_F;
    if (j < p.N1) {
      y0[t] = __ldg(gy + (size_t)j * 3);
      y1[t] = __ldg(gy + (size_t)j * 3 + 1);
      y2[t] = __ldg(gy + (size_t)j * 3 + 2);
      ry[t] = hg_dot3_fma(y0[t], y1[t], y2[t], y0[t], y1[t], y2[t]);
    }
  }
  __syncthreads();

  if (warp_active) {
    float cm[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
      cm[t] = CUDART_INF_F;
      sprev[t * WARPS * 32 + threadIdx.x] = CUDART_INF_F;
      scid[t * WARPS * 32 + threadIdx.x] = r0 / kColBatch;
    }
    uint4 *myrow = rowpart + (size_t)warp * (p.RB / 2);

    // Packed FP32 over ROW pairs: each FMUL2/FFMA2/FADD2 produces (P[a][t], P[b][t]) for one column t.  The row
    // operands (X0,X1,X2,RX) are shared by T consecutive instructions, which is what lets the operand-reuse
    // cache absorb one of the two 64-bit register reads (ptxas flags ~75% of the FFMA2s; with the columns packed
    // instead it flags ~18% and the pipe issues every 3rd cycle).  Four rows per iteration.
    float4 xA = xs[0], xB = xs[1], xC = xs[2], xD = xs[3];
    for (int rb = 0; rb < p.RB; rb += kColBatch) {
#pragma unroll 2
      for (int rr = 0; rr < kColBatch; rr += 4) {
        const int rq = (rb + rr) >> 1;  // row pair index
        const float4 nA = xs[2 * rq + 4], nB = xs[2 * rq + 5], nC = xs[2 * rq + 6], nD = xs[2 * rq + 7];
        const float2 X0 = make_float2(xA.x, xA.y), X1 = make_float2(xA.z, xA.w), X2 = make_float2(xB.x, xB.y),
                     RX = make_float2(xB.z, xB.w);
        const float2 Z0 = make_float2(xC.x, xC.y), Z1 = make_float2(xC.z, xC.w), Z2 = make_float2(xD.x, xD.y),
                     RZ = make_float2(xD.z, xD.w);
        float2 P[T], Q[T];
#pragma unroll
        for (int t = 0; t < T; ++t) {
          float2 tt = __fmul2_rn(make_float2(y0[t], y0[t]), X0);
          float2 uu = __fmul2_rn(make_float2(y0[t], y0[t]), Z0);
          tt = __ffma2_rn(make_float2(y1[t], y1[t]), X1, tt);
          uu = __ffma2_rn(make_float2(y1[t], y1[t]), Z1, uu);
          tt = __ffma2_rn(make_float2(y2[t], y2[t]), X2, tt);
          uu = __ffma2_rn(make_float2(y2[t], y2[t]), Z2, uu);
          P[t] = __fadd2_rn(__fadd2_rn(RX, make_float2(ry[t], ry[t])), tt);  // (rx + ry) + zz'
          Q[t] = __fadd2_rn(__fadd2_rn(RZ, make_float2(ry[t], ry[t])), uu);
          cm[t] = fminf(fminf(fminf(fminf(cm[t], P[t].x), P[t].y), Q[t].x), Q[t].y);  // 2 x FMNMX3
        }
        float ma = fminf(P[0].x, P[1].x), mb = fminf(P[0].y, P[1].y);
        float mc = fminf(Q[0].x, Q[1].x), md = fminf(Q[0].y, Q[1].y);
#pragma unroll
        for (int t = 2; t < T; t += 2) {
          ma = fminf(fminf(ma, P[t].x), P[t + 1].x);
          mb = fminf(fminf(mb, P[t].y), P[t + 1].y);
          mc = fminf(fminf(mc, Q[t].x), Q[t + 1].x);
          md = fminf(fminf(md, Q[t].y), Q[t + 1].y);
        }
        const float wa = hg_warp_min_f32(ma), wb = hg_warp_min_f32(mb);
        const float wc = hg_warp_min_f32(mc), wd = hg_warp_min_f32(md);
        const unsigned ka = __ballot_sync(0xffffffffu, ma == wa), kb = __ballot_sync(0xffffffffu, mb == wb);
        const unsigned kc = __ballot_sync(0xffffffffu, mc == wc), kd = __ballot_sync(0xffffffffu, md == wd);
        if (lane == 0) {
          myrow[rq] = make_uint4(__float_as_uint(wa), ka, __float_as_uint(wb), kb);
          myrow[rq + 1] = make_uint4(__float_as_uint(wc), kc, __float_as_uint(wd), kd);
        }
        xA = nA;
        xB = nB;
        xC = nC;
        xD = nD;
      }
      const int batch = (r0 + rb) / kColBatch;
#pragma unroll
      for (int t = 0; t < T; ++t) {
        if (cm[t] < sprev[t * WARPS * 32 + threadIdx.x]) scid[t * WARPS * 32 + threadIdx.x] = batch;
        sprev[t * WARPS * 32 + threadIdx.x] = cm[t];
      }
    }
    // column direction: merge with the other row blocks
    unsigned long long *cr = p.colres + (size_t)b * p.N1;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int j = cbase + t;
      if (j < p.N1)
        atomicMin(cr + j, ((unsigned long long)hg_ord(cm[t]) << 32) | (unsigned)scid[t * WARPS * 32 + threadIdx.x]);
    }
  }
  __syncthreads();

  // row direction: merge the CTA's warps (lowest warp = lowest columns wins ties), then the other CTAs
  unsigned long long *rr_out = p.rowres + (size_t)b * p.N2;
  for (int r = threadIdx.x; r < p.RB; r += WARPS * 32) {
    const int i = r0 + r;
    if (i >= p.N2) continue;
    float best = CUDART_INF_F;
    unsigned code = 0xffffffffu;
    for (int w = 0; w < WARPS; ++w) {
      if ((blockIdx.y * WARPS + w) * 32 * T >= p.N1) break;
      const uint4 v = rowpart[(size_t)w * (p.RB / 2) + (r >> 1)];
      const float m = __uint_as_float((r & 1) ? v.z : v.x);
      const unsigned mask = (r & 1) ? v.w : v.y;
      const unsigned c = ((unsigned)(blockIdx.y * WARPS + w) << 5) | (unsigned)(__ffs(mask) - 1);
      if (m < best || code == 0xffffffffu) {
        best = m;
        code = c;
      }
    }
    atomicMin(rr_out + i, ((unsigned long long)hg_ord(best) << 32) | code);
  }
}

// Exact first-index recovery (torch.min tie rule) + unpacking of the merged results.
template <int T>
__global__ void __launch_bounds__(256) nn_bidir_d3_finish_kernel(NnParams p, int B, float *__restrict__ min1,
                                                                  int *__restrict__ arg1, float *__restrict__ min2,
                                                                  int *__restrict__ arg2) {
  const long long total = (long long)B * (p.N1 + p.N2);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(g / (p.N1 + p.N2));
    const int e = (int)(g % (p.N1 + p.N2));
    if (nn_skip(p, b)) continue;
    const float *gx = p.gts + (size_t)b * p.N2 * 3;
    const float *gy = p.preds + (size_t)b * p.N1 * 3;
    if (e < p.N1) {  // column j: nearest row inside the recorded batch of kColBatch rows
      const int j = e;
      const unsigned long long key = p.colres[(size_t)b * p.N1 + j];
      const float m = hg_unord((unsigned)(key >> 32));
      const int i0 = (int)(unsigned)(key & 0xffffffffu) * kColBatch;
      const float y0 = __ldg(gy + (size_t)j * 3), y1 = __ldg(gy + (size_t)j * 3 + 1), y2 = __ldg(gy + (size_t)j * 3 + 2);
      int arg = 0;
      bool found = false;
#pragma unroll
      for (int d = 0; d < kColBatch; ++d) {
        const int i = i0 + d;
        if (i < p.N2 && !found) {
          const float v = nn_p_exact(__ldg(gx + (size_t)i * 3), __ldg(gx + (size_t)i * 3 + 1),
                                     __ldg(gx + (size_t)i * 3 + 2), y0, y1, y2);
          if (v == m) {
            arg = i;
            found = true;
          }
        }
      }
      min1[(size_t)b * p.N1 + j] = m;
      arg1[(size_t)b * p.N1 + j] = arg;
    } else {  // row i: nearest column among the T columns of the recorded lane
      const int i = e - p.N1;
      const unsigned long long key = p.rowres[(size_t)b * p.N2 + i];
      const float m = hg_unord((unsigned)(key >> 32));
      const unsigned code = (unsigned)(key & 0xffffffffu);
      const int j0 = (int)(code >> 5) * 32 * T + (int)(code & 31u) * T;
      const float x0 = __ldg(gx + (size_t)i * 3), x1 = __ldg(gx + (size_t)i * 3 + 1), x2 = __ldg(gx + (size_t)i * 3 + 2);
      int arg = 0;
      bool found = false;
#pragma unroll
      for (int d = 0; d < T; ++d) {
        const int j = j0 + d;
        if (j < p.N1 && !found) {
          const float v = nn_p_exact(x0, x1, x2, __ldg(gy + (size_t)j * 3), __ldg(gy + (size_t)j * 3 + 1),
                                     __ldg(gy + (size_t)j * 3 + 2));
          if (v == m) {
            arg = j;
            found = true;
          }
        }
      }
      min2[(size_t)b * p.N2 + i] = m;
      arg2[(size_t)b * p.N2 + i] = arg;
    }
  }
}

// Small clouds (each fits in shared memory): a CTA stages ONE cloud as padded structure-of-arrays and re-scans either
// 256 column entries against the rows (the 32-row batch of an entry split over FOUR lanes, 8 rows each, first match per
// lane, quad minimum) or 1024 row entries against the columns (T columns per entry): 8 or T evaluations per thread and
// iteration, four iterations, the four keys loaded up front.  The gather version above issues up to 96 scalar global
// loads per column entry and is latency-bound at 1024 points (26 us at 388 x 1024, a quarter of the main kernel).
// Same arithmetic, same first-index rule.
constexpr int kFinColsPerCta = 256, kFinRowsPerCta = 1024;

template <int T>
__global__ void __launch_bounds__(256) nn_bidir_d3_finish_small_kernel(NnParams p, int ncolcta, float *__restrict__ min1,
                                                                        int *__restrict__ arg1, float *__restrict__ min2,
                                                                        int *__restrict__ arg2) {
  constexpr int kTShift = T == 16 ? 4 : 3;
  extern __shared__ float fsm[];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int N1 = p.N1, N2 = p.N2;
  if (nn_skip(p, b)) return;
  const float *gx = p.gts + (size_t)b * N2 * 3;
  const float *gy = p.preds + (size_t)b * N1 * 3;
  if ((int)blockIdx.y < ncolcta) {
    // rows staged; pad one slot per 32 (a quad walks the rows of ITS batch; batches differ between quads)
    const int xs = N2 + (N2 >> 5) + 1;
    float *sx0 = fsm, *sx1 = fsm + xs, *sx2 = fsm + 2 * xs;
    const int jbase = blockIdx.y * kFinColsPerCta;
    unsigned long long key[4];
    float y0[4], y1[4], y2[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int j = jbase + ((it * 256 + tid) >> 2);
      key[it] = 0ull;
      y0[it] = y1[it] = y2[it] = 0.f;
      if (j < N1) {
        key[it] = p.colres[(size_t)b * N1 + j];
        y0[it] = __ldg(gy + (size_t)j * 3);
        y1[it] = __ldg(gy + (size_t)j * 3 + 1);
        y2[it] = __ldg(gy + (size_t)j * 3 + 2);
      }
    }
    for (int q = tid; q < N2 * 3; q += 256) {
      const int i = q / 3, c = q - 3 * i;
      fsm[c * xs + i + (i >> 5)] = __ldg(gx + q);
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int u = it * 256 + tid, j = jbase + (u >> 2), part = u & 3;
      const bool live = j < N1;
      const float m = hg_unord((unsigned)(key[it] >> 32));
      int arg = 0x7fffffff;
      if (live) {
        const int i0 = (int)(unsigned)(key[it] & 0xffffffffu) * kColBatch + part * 8;
#pragma unroll
        for (int d = 7; d >= 0; --d) {  // descending: the smallest matching row is what stays
          const int i = i0 + d;
          if (i < N2) {
            const int ii = i + (i >> 5);
            if (nn_p_exact(sx0[ii], sx1[ii], sx2[ii], y0[it], y1[it], y2[it]) == m) arg = i;
          }
        }
      }
      arg = min(arg, __shfl_xor_sync(0xffffffffu, arg, 1));
      arg = min(arg, __shfl_xor_sync(0xffffffffu, arg, 2));
      if (live && part == 0) {
        min1[(size_t)b * N1 + j] = m;
        arg1[(size_t)b * N1 + j] = arg == 0x7fffffff ? 0 : arg;
      }
    }
  } else {
    // columns staged; pad one slot per T (a row entry walks the T columns of its lane; lanes differ by T)
    const int ys = N1 + (N1 >> kTShift) + 1;
    float *sy0 = fsm, *sy1 = fsm + ys, *sy2 = fsm + 2 * ys;
    const int ibase = ((int)blockIdx.y - ncolcta) * kFinRowsPerCta;
    unsigned long long key[4];
    float x0[4], x1[4], x2[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int i = ibase + it * 256 + tid;
      key[it] = 0ull;
      x0[it] = x1[it] = x2[it] = 0.f;
      if (i < N2) {
        key[it] = p.rowres[(size_t)b * N2 + i];
        x0[it] = __ldg(gx + (size_t)i * 3);
        x1[it] = __ldg(gx + (size_t)i * 3 + 1);
        x2[it] = __ldg(gx + (size_t)i * 3 + 2);
      }
    }
    for (int q = tid; q < N1 * 3; q += 256) {
      const int j = q / 3, c = q - 3 * j;
      fsm[c * ys + j + (j >> kTShift)] = __ldg(gy + q);
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int i = ibase + it * 256 + tid;
      if (i >= N2) continue;
      const float m = hg_unord((unsigned)(key[it] >> 32));
      const unsigned code = (unsigned)(key[it] & 0xffffffffu);
      const int j0 = (int)(code >> 5) * 32 * T + (int)(code & 31u) * T;
      int arg = 0;
#pragma unroll
      for (int d = T - 1; d >= 0; --d) {
        const int j = j0 + d;
        if (j < N1) {
          const int jj = j + (j >> kTShift);
          if (nn_p_exact(x0[it], x1[it], x2[it], sy0[jj], sy1[jj], sy2[jj]) == m) arg = j;
        }
      }
      min2[(size_t)b * N2 + i] = m;
      arg2[(size_t)b * N2 + i] = arg;
    }
  }
}

template <int T>
static int launch_finish_small(const NnParams &p, int B, float *min1, int *arg1, float *min2, int *arg2, size_t smem,
                               cudaStream_t stream) {
  static HgPerDeviceOnce once;
  if (once.first())
    HG_CUDA(cudaFuncSetAttribute(nn_bidir_d3_finish_small_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 kFinishSmallSmemMax));
  const int ncol = (p.N1 + kFinColsPerCta - 1) / kFinColsPerCta, nrow = (p.N2 + kFinRowsPerCta - 1) / kFinRowsPerCta;
  nn_bidir_d3_finish_small_kernel<T><<<dim3(B, ncol + nrow), 256, smem, stream>>>(p, ncol, min1, arg1, min2, arg2);
  HG_CHECK_LAUNCH("nn_bidir_d3_finish_small_kernel");
  return HG_OK;
}

// ---- generic inner dimension (R3: HiT_ADV.py:229-231 feeds [B,3,K], i.e. N=3 "points" of dimension K) ------
// One thread per matrix entry, sequential FMA chain over D (the order the oracle uses).  Small problems only.
__global__ void nn_generic_p_kernel(const float *__restrict__ gts, const float *__restrict__ preds, int B, int N2,
                                    int N1, int D, float *__restrict__ P) {
  const long long total = (long long)B * N2 * N1;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(g % N1);
    const int i = (int)((g / N1) % N2);
    const int b = (int)(g / ((long long)N1 * N2));
    const float *x = gts + ((size_t)b * N2 + i) * D;
    const float *y = preds + ((size_t)b * N1 + j) * D;
    float rx = __fmul_rn(x[0], x[0]), ry = __fmul_rn(y[0], y[0]), zz = __fmul_rn(x[0], y[0]);
    for (int c = 1; c < D; ++c) {
      const float xc = x[c], yc = y[c];
      rx = __fmaf_rn(xc, xc, rx);
      ry = __fmaf_rn(yc, yc, ry);
      zz = __fmaf_rn(xc, yc, zz);
    }
    P[g] = __fsub_rn(__fadd_rn(rx, ry), __fmul_rn(2.0f, zz));
  }
}

__global__ void nn_generic_min_kernel(const float *__restrict__ P, int B, int N2, int N1, float *__restrict__ min1,
                                      int *__restrict__ arg1, float *__restrict__ min2, int *__restrict__ arg2) {
  const long long total = (long long)B * (N1 + N2);
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(g / (N1 + N2));
    const int e = (int)(g % (N1 + N2));
    const float *Pb = P + (size_t)b * N2 * N1;
    float best = CUDART_INF_F;
    int arg = 0;
    if (e < N1) {
      for (int i = 0; i < N2; ++i) {
        const float v = Pb[(size_t)i * N1 + e];
        if (v < best) {
          best = v;
          arg = i;
        }
      }
      min1[(size_t)b * N1 + e] = best;
      arg1[(size_t)b * N1 + e] = arg;
    } else {
      const int i = e - N1;
      for (int j = 0; j < N1; ++j) {
        const float v = Pb[(size_t)i * N1 + j];
        if (v < best) {
          best = v;
          arg = j;
        }
      }
      min2[(size_t)b * N2 + i] = best;
      arg2[(size_t)b * N2 + i] = arg;
    }
  }
}

// ---- Chamfer mean / Hausdorff max over the mins (set_distance.py:46-49, :66-69) -----------------------------
// One CTA per (cloud, direction); fixed-order tree => deterministic.
__global__ void __launch_bounds__(256) set_loss_kernel(const float *__restrict__ min1, const float *__restrict__ min2,
                                                       int N1, int N2, int mode, float *__restrict__ loss1,
                                                       float *__restrict__ loss2, int *__restrict__ hd_arg1,
                                                       int *__restrict__ hd_arg2) {
  const int b = blockIdx.x, dir = blockIdx.y;
  const int N = dir ? N2 : N1;
  const float *m = (dir ? min2 : min1) + (size_t)b * N;
  __shared__ double sh_sum[256];
  __shared__ float sh_val[256];
  __shared__ int sh_idx[256];
  const int tid = threadIdx.x;
  if (mode == HG_MODE_CHAMFER) {
    double s = 0.0;
    for (int i = tid; i < N; i += 256) s += (double)m[i];
    sh_sum[tid] = s;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
      if (tid < st) sh_sum[tid] += sh_sum[tid + st];
      __syncthreads();
    }
    if (tid == 0) (dir ? loss2 : loss1)[b] = (float)(sh_sum[0] / (double)N);
  } else {
    float v = -CUDART_INF_F;
    int a = 0x7fffffff;
    for (int i = tid; i < N; i += 256) {
      const float x = m[i];
      if (x > v) {  // ascending i per thread: strict '>' keeps the first
        v = x;
        a = i;
      }
    }
    sh_val[tid] = v;
    sh_idx[tid] = a;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
      if (tid < st) {
        const float v2 = sh_val[tid + st];
        const int a2 = sh_idx[tid + st];
        if (v2 > sh_val[tid] || (v2 == sh_val[tid] && a2 < sh_idx[tid])) {
          sh_val[tid] = v2;
          sh_idx[tid] = a2;
        }
      }
      __syncthreads();
    }
    if (tid == 0) {
      (dir ? loss2 : loss1)[b] = sh_val[0];
      int *ha = dir ? hd_arg2 : hd_arg1;
      if (ha) ha[b] = sh_idx[0] == 0x7fffffff ? 0 : sh_idx[0];
    }
  }
}

// ---- backward ---------------------------------------------------------------------------------------------
// dP[i,j]/dy_j = 2(y_j - x_i), dP[i,j]/dx_i = 2(x_i - y_j).
//   chamfer:  grad_y[j] = (g1/N1) 2(y_j - x_{arg1[j]})  +  (g2/N2) sum_{i: arg2[i]==j} 2(y_j - x_i)
//             grad_x[i] = (g2/N2) 2(x_i - y_{arg2[i]})  +  (g1/N1) sum_{j: arg1[j]==i} 2(x_i - y_j)
//   hausdorff: the same with one-hot row weights (only the arg-max pair of each direction).
// The sums run over the reverse map in ascending source index: deterministic, no float atomics.
__global__ void __launch_bounds__(256) set_loss_bwd_kernel(
    const float *__restrict__ self_pts /*[B,Ns,D] points receiving the gradient*/,
    const float *__restrict__ other_pts /*[B,No,D]*/, const int *__restrict__ self_arg /*[B,Ns] -> other*/,
    const int *__restrict__ rev_off /*[B,Ns+1]*/, const int *__restrict__ rev_list /*[B,No] other idx, any order*/,
    const int *__restrict__ other_arg /*[B,No] -> self: the map rev_off/rev_list inverts*/,
    const float *__restrict__ g_self /*[B] upstream of the loss that gathers (self -> nearest other)*/,
    const float *__restrict__ g_other /*[B] upstream of the loss that scatters into self*/,
    const int *__restrict__ hd_self /*[B] or null*/, const int *__restrict__ hd_other /*[B] or null*/, int B, int Ns,
    int No, int D, int mode, float *__restrict__ grad_self) {
  // D == 3 (the hot case): one thread per point, looping over its 3 coordinates.  Large D (channel-first input,
  // SURVEY.md R3: 3 "points" of dimension K): one thread per (point, coordinate) so that loads/stores coalesce.
  const int cper = (D > 8) ? 1 : D;          // coordinates handled per thread
  const int nchunk = (D + cper - 1) / cper;  // threads per point
  const long long total = (long long)B * Ns * nchunk;
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const int chunk = (int)(g % nchunk);
    const long long pt = g / nchunk;
    const int b = (int)(pt / Ns), s = (int)(pt % Ns);
    const float *ps = self_pts + ((size_t)b * Ns + s) * D;
    const float *po = other_pts + (size_t)b * No * D;
    float cs, co;
    // a null upstream = that loss is unused (ChamferDist's default 'adv2ori' never touches loss2): its term is
    // skipped, and the host did not even build the reverse map (rev_off == nullptr)
    const float gs = g_self ? g_self[b] : 0.f, go = g_other ? g_other[b] : 0.f;
    if (mode == HG_MODE_CHAMFER) {
      cs = gs / (float)Ns;
      co = go / (float)No;
    } else {
      cs = (hd_self[b] == s) ? gs : 0.f;
      co = go;
    }
    const int a = self_arg[(size_t)b * Ns + s];
    const int *off = rev_off ? rev_off + (size_t)b * (Ns + 1) : nullptr;
    const int *lst = rev_list + (size_t)b * No;
    const int p0 = off ? off[s] : 0, p1 = off ? off[s + 1] : 0;
    const int hdo = (mode == HG_MODE_CHAMFER) ? -1 : hd_other[b];
    for (int c = chunk * cper; c < min(D, (chunk + 1) * cper); ++c) {
      const float v = ps[c];
      float acc = 0.f;
      if (cs != 0.f) acc = cs * (2.0f * (v - po[(size_t)a * D + c]));
      float sc = 0.f;
      if (p1 - p0 <= kCsrWalkMax) {
        int o = -1;
        for (int q = p0; q < p1; ++q) {  // ascending source index, whatever order the list was filled in
          o = hg_csr_next(lst, p0, p1, o);
          if (mode == HG_MODE_CHAMFER || o == hdo) sc += 2.0f * (v - po[(size_t)o * D + c]);
        }
      } else {
        // a hub (collapsed / duplicated points: hundreds of sources share this nearest neighbour): the selection walk
        // above is O(deg^2); scanning the forward map in ascending source order is O(No) and sums in the same order
        const int *oa = other_arg + (size_t)b * No;
        for (int o = 0; o < No; ++o)
          if (oa[o] == s && (mode == HG_MODE_CHAMFER || o == hdo)) sc += 2.0f * (v - po[(size_t)o * D + c]);
      }
      grad_self[((size_t)b * Ns + s) * D + c] = acc + co * sc;
    }
  }
}

template <int T, int WARPS>
int launch_main(const NnParams &p, int B, cudaStream_t stream) {
  const int ncg = (p.N1 + 32 * T - 1) / (32 * T);
  dim3 grid((p.N2 + p.RB - 1) / p.RB, (ncg + WARPS - 1) / WARPS, B);
  const size_t smem = (size_t)(p.RB + 4) * sizeof(float4) + (size_t)WARPS * (p.RB / 2) * sizeof(uint4) +
                      (size_t)2 * T * WARPS * 32 * sizeof(float);
  auto kernel = nn_bidir_d3_kernel<T, WARPS>;
  if (smem > 48 * 1024) {
    HG_REQUIRE(smem <= 200 * 1024, HG_E_UNSUPPORTED, "nn_bidir: RB=%d needs %zu bytes of shared memory", p.RB, smem);
    HG_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  const bool prof = hg_prof_begin(HG_PROF_NN_BIDIR, stream);
  kernel<<<grid, WARPS * 32, smem, stream>>>(p);
  hg_prof_end(HG_PROF_NN_BIDIR, stream, prof);
  HG_CHECK_LAUNCH("nn_bidir_d3_kernel");
  return HG_OK;
}

template <int T>
int launch_warps(const NnParams &p, int B, int ncg, cudaStream_t stream) {
  return (ncg >= 4 && ncg % 4 == 0) ? launch_main<T, 4>(p, B, stream)
         : (ncg >= 2)               ? launch_main<T, 2>(p, B, stream)
                                    : launch_main<T, 1>(p, B, stream);
}

}  // namespace

// Tunables exposed for the benchmark sweep (not part of the stable ABI): T (columns per lane: 8 or 16) and
// rows per CTA.  0 = automatic.
static int g_force_T = 0, g_force_RB = 0;
int g_hg_tune_small_fused_off = 0;
HG_API void hg_nn_bidir_tune(int T, int RB) {
  g_force_T = T;
  g_force_RB = RB;
}

// D = 3: merged (value, cell) keys of both directions (the part each call resets to 0xff), a reserved region, then the
// kd-tree orderings of both clouds (0 bytes where the pruned path does not apply)
struct NnD3Workspace {
  size_t keys_bytes;
  void *gts_order, *preds_order;
  NnD3Workspace(HgCarve &c, int B, int N2, int N1, NnParams *p) {
    p->colres = c.take<unsigned long long>((size_t)B * N1);
    p->rowres = c.take<unsigned long long>((size_t)B * N2);
    keys_bytes = c.bytes;
    // unused: keeps hg_nn_bidir_workspace_bytes at the sizes tests/test_cpu_workspace_sizes.py pins as C ABI
    c.take<char>(hg_align((size_t)B * N1 * 4) + hg_align((size_t)B * N2 * 4) + hg_align((size_t)B * 4) +
                 hg_align(((size_t)B * (N1 + N2) + 1) * 4));
    gts_order = c.span(hg_prune_order_bytes(B, N2)).ptr;
    preds_order = c.span(hg_prune_order_bytes(B, N1)).ptr;
  }
};
struct NnGenericWorkspace {  // other D: P [B,N2,N1]
  float *P;
  NnGenericWorkspace(HgCarve &c, int B, int N2, int N1) : P(c.take<float>((size_t)B * N2 * N1)) {}
};

HG_API size_t hg_nn_bidir_workspace_bytes(int B, int N2, int N1, int D) {
  if (B <= 0 || N1 <= 0 || N2 <= 0 || D <= 0) return 0;
  NnParams p;
  return D == 3 ? hg_layout_bytes<NnD3Workspace>(B, N2, N1, &p) : hg_layout_bytes<NnGenericWorkspace>(B, N2, N1);
}

HG_API int hg_nn_bidir_f32(const float *gts, const float *preds, int B, int N2, int N1, int D, float *min1, int *arg1,
                           float *min2, int *arg2, void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_nn_bidir_f32");
  return hg_nn_bidir_temporal_f32(gts, preds, B, N2, N1, D, min1, arg1, min2, arg2, nullptr, nullptr, workspace,
                                  workspace_bytes, stream_);
}

HG_API int hg_nn_bidir_temporal_f32(const float *gts, const float *preds, int B, int N2, int N1, int D, float *min1,
                                    int *arg1, float *min2, int *arg2, void *gts_order, void *preds_order,
                                    void *workspace, size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_nn_bidir_temporal_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(gts && preds && min1 && arg1 && min2 && arg2, HG_E_BADARG, "nn_bidir: null pointer");
  HG_REQUIRE(((uintptr_t)gts_order & 15) == 0 && ((uintptr_t)preds_order & 15) == 0, HG_E_BADARG,
             "nn_bidir: ordering states must be 16-byte aligned");
  HG_REQUIRE(gts_order == nullptr || gts_order != preds_order, HG_E_BADARG,
             "nn_bidir: gts and preds need ordering states of their own");
  HG_REQUIRE(B > 0 && N1 > 0 && N2 > 0 && D > 0, HG_E_BADARG, "nn_bidir: sizes must be positive (B=%d N2=%d N1=%d D=%d)",
             B, N2, N1, D);
  HG_REQUIRE(B <= 65535, HG_E_UNSUPPORTED, "nn_bidir: B=%d > 65535 clouds per call", B);
  const size_t need = hg_nn_bidir_workspace_bytes(B, N2, N1, D);
  HG_REQUIRE(workspace && workspace_bytes >= need, HG_E_WORKSPACE, "nn_bidir: workspace too small (%zu < %zu)",
             workspace_bytes, need);
  if (D != 3) {
    HG_REQUIRE((double)B * N2 * N1 <= 2.0e9, HG_E_UNSUPPORTED,
               "nn_bidir: generic-D path materialises P; B*N2*N1 too large");
    float *P = hg_layout_at<NnGenericWorkspace>(workspace, B, N2, N1).P;
    const long long total = (long long)B * N2 * N1;
    nn_generic_p_kernel<<<hg_grid_for(total, 256, 16), 256, 0, stream>>>(gts, preds, B, N2, N1, D, P);
    HG_CHECK_LAUNCH("nn_generic_p_kernel");
    nn_generic_min_kernel<<<hg_grid_for((long long)B * (N1 + N2), 128, 16), 128, 0, stream>>>(P, B, N2, N1, min1, arg1, min2,
                                                                                                arg2);
    HG_CHECK_LAUNCH("nn_generic_min_kernel");
    return HG_OK;
  }
  NnParams p;
  p.gts = gts;
  p.preds = preds;
  p.N2 = N2;
  p.N1 = N1;
  const auto w = hg_layout_at<NnD3Workspace>(workspace, B, N2, N1, &p);
  p.only_a = p.only_b = nullptr;
  // large clouds: kd-tree orderings and pruned 1-NN passes in both directions (hg_prune.cu); the all-pairs kernels below
  // then run on the clouds the ordering build flagged (non-finite coordinates) only
  const bool prune = hg_prune_applies(N1) && hg_prune_applies(N2);
  if (prune) {
    HgPruneOrder og, op;
    const bool prof = hg_prof_begin(HG_PROF_NN_BIDIR, stream);
    int rc = hg_prune_build(gts, B, N2, true, w.gts_order, &og, stream, gts_order);
    if (!rc) rc = hg_prune_build(preds, B, N1, true, w.preds_order, &op, stream, preds_order);
    if (!rc) rc = hg_prune_nn_search(op, og, B, min1, arg1, stream);  // column j (preds): nearest row (gts)
    if (!rc) rc = hg_prune_nn_search(og, op, B, min2, arg2, stream);  // row i (gts): nearest column (preds)
    hg_prof_end(HG_PROF_NN_BIDIR, stream, prof);
    if (rc) return rc;
    p.only_a = og.info;
    p.only_b = op.info;
  }
  HG_CUDA(cudaMemsetAsync(workspace, 0xff, w.keys_bytes, stream));

  // columns per lane: 16 halves the row broadcasts per pair but needs 12-warp occupancy to pay (tools/debug/nn_sweep.py,
  // B200: 8 wins by 6 % at 2048 points, 2 % at 4096, level at 8192, loses from there)
  int T = g_force_T ? g_force_T : (N1 >= 8192 ? 16 : 8);
  // rows per CTA: amortise the per-CTA column load and result merge (measured: >= 128 rows is flat, 64 costs
  // ~4-10 %, 32 more), but keep several waves of CTAs on the machine
  int RB = g_force_RB;
  if (!RB) {
    const int ncg_ = (N1 + 32 * T - 1) / (32 * T);
    const int wpc = (ncg_ >= 4 && ncg_ % 4 == 0) ? 4 : (ncg_ >= 2 ? 2 : 1);
    RB = 1024;  // (256 x 16384: 14.25 ms with 1024 rows per CTA, 14.33 with 512, 14.66 with 256)
    while (RB > 2 * kColBatch) {
      const long long ctas = (long long)B * ((N2 + RB - 1) / RB) * ((ncg_ + wpc - 1) / wpc);
      if (ctas * wpc >= (long long)hg_sm_count() * 12 * 4) break;  // >= 4 waves of 12 warps per SM
      RB >>= 1;
    }
    if (RB > N2) RB = (N2 + kColBatch - 1) / kColBatch * kColBatch;
  }
  RB = (RB + kColBatch - 1) / kColBatch * kColBatch;
  if (RB > 1024) RB = 1024;
  p.RB = RB;
  if (T != 16) T = 8;
  const int ncg = (N1 + 32 * T - 1) / (32 * T);
  const int rc = T == 16 ? launch_warps<16>(p, B, ncg, stream) : launch_warps<8>(p, B, ncg, stream);
  if (rc) return rc;
  const long long total = (long long)B * (N1 + N2);
  {
    const int tshift = T == 16 ? 4 : 3;
    const size_t sx = (size_t)(N2 + (N2 >> 5) + 1), sy = (size_t)(N1 + (N1 >> tshift) + 1);
    const size_t smem = 3 * (sx > sy ? sx : sy) * sizeof(float);
    if (smem <= (size_t)kFinishSmallSmemMax && B <= 65535 && !g_hg_tune_small_fused_off)
      return T == 16 ? launch_finish_small<16>(p, B, min1, arg1, min2, arg2, smem, stream)
                     : launch_finish_small<8>(p, B, min1, arg1, min2, arg2, smem, stream);
  }
  if (T == 16)
    nn_bidir_d3_finish_kernel<16><<<hg_grid_for(total, 256, 16), 256, 0, stream>>>(p, B, min1, arg1, min2, arg2);
  else
    nn_bidir_d3_finish_kernel<8><<<hg_grid_for(total, 256, 16), 256, 0, stream>>>(p, B, min1, arg1, min2, arg2);
  HG_CHECK_LAUNCH("nn_bidir_d3_finish_kernel");
  return HG_OK;
}

HG_API int hg_pairwise_dist_f32(const float *x, const float *y, int B, int Nx, int Ny, int D, float *P,
                                hgStream stream_) {
  HG_NVTX_RANGE("hg_pairwise_dist_f32");
  HG_REQUIRE(x && y && P, HG_E_BADARG, "pairwise_dist: null pointer");
  HG_REQUIRE(B > 0 && Nx > 0 && Ny > 0 && D > 0, HG_E_BADARG, "pairwise_dist: sizes must be positive");
  const long long total = (long long)B * Nx * Ny;
  nn_generic_p_kernel<<<hg_grid_for(total, 256, 16), 256, 0, hg_stream(stream_)>>>(x, y, B, Nx, Ny, D, P);
  HG_CHECK_LAUNCH("nn_generic_p_kernel");
  return HG_OK;
}

HG_API int hg_set_loss_f32(const float *min1, const float *min2, int B, int N1, int N2, int mode, float *loss1,
                           float *loss2, int *hd_arg1, int *hd_arg2, hgStream stream_) {
  HG_NVTX_RANGE("hg_set_loss_f32");
  HG_REQUIRE(min1 && min2 && loss1 && loss2, HG_E_BADARG, "set_loss: null pointer");
  HG_REQUIRE(B > 0 && N1 > 0 && N2 > 0, HG_E_BADARG, "set_loss: sizes must be positive");
  HG_REQUIRE(mode == HG_MODE_CHAMFER || mode == HG_MODE_HAUSDORFF, HG_E_BADARG, "set_loss: bad mode %d", mode);
  set_loss_kernel<<<dim3(B, 2), 256, 0, hg_stream(stream_)>>>(min1, min2, N1, N2, mode, loss1, loss2, hd_arg1, hd_arg2);
  HG_CHECK_LAUNCH("set_loss_kernel");
  return HG_OK;
}

// reverse map of arg2 (N2 edges -> N1 keys), then of arg1 (N1 edges -> N2 keys)
struct SetLossBwdWorkspace {
  HgSpan rev2, rev1;
  SetLossBwdWorkspace(HgCarve &c, int B, int N2, int N1)
      : rev2(c.span(hg_csr_workspace_bytes(B, N1, N2))), rev1(c.span(hg_csr_workspace_bytes(B, N2, N1))) {}
};

HG_API size_t hg_set_loss_bwd_workspace_bytes(int B, int N2, int N1) {
  if (B <= 0 || N1 <= 0 || N2 <= 0) return 0;
  return hg_layout_bytes<SetLossBwdWorkspace>(B, N2, N1);
}

HG_API int hg_set_loss_bwd_f32(const float *gts, const float *preds, const int *arg1, const int *arg2,
                               const int *hd_arg1, const int *hd_arg2, const float *g1, const float *g2, int B, int N2,
                               int N1, int D, int mode, float *grad_preds, float *grad_gts, void *workspace,
                               size_t workspace_bytes, hgStream stream_) {
  HG_NVTX_RANGE("hg_set_loss_bwd_f32");
  cudaStream_t stream = hg_stream(stream_);
  HG_REQUIRE(gts && preds && arg1 && arg2 && grad_preds, HG_E_BADARG, "set_loss_bwd: null pointer");
  HG_REQUIRE(g1 || g2, HG_E_BADARG, "set_loss_bwd: g1 and g2 are both null (nothing to differentiate)");
  HG_REQUIRE(B > 0 && N1 > 0 && N2 > 0 && D > 0, HG_E_BADARG, "set_loss_bwd: sizes must be positive");
  HG_REQUIRE(mode == HG_MODE_CHAMFER || (mode == HG_MODE_HAUSDORFF && hd_arg1 && hd_arg2), HG_E_BADARG,
             "set_loss_bwd: bad mode / missing hausdorff arg-max indices");
  HG_REQUIRE(workspace && workspace_bytes >= hg_set_loss_bwd_workspace_bytes(B, N2, N1), HG_E_WORKSPACE,
             "set_loss_bwd: workspace too small");
  const auto w = hg_layout_at<SetLossBwdWorkspace>(workspace, B, N2, N1);
  // preds (adv, "y"): gathers through arg1 (loss1), receives scatter from arg2 (loss2)
  HgCsr rev2;
  int rc = HG_OK;
  rev2.off = nullptr;
  rev2.list = nullptr;
  if (g2) {  // loss2 scatters into preds through arg2; unused (g2 == NULL) => no reverse map at all
    rc = hg_csr_build_unordered(arg2, B, N2, N1, w.rev2.ptr, w.rev2.bytes, &rev2, stream);
    if (rc) return rc;
  }
  const long long tp = (long long)B * N1 * (D > 8 ? D : 1);
  set_loss_bwd_kernel<<<hg_grid_for(tp, 256, 16), 256, 0, stream>>>(preds, gts, arg1, rev2.off, rev2.list, arg2, g1, g2,
                                                                    hd_arg1, hd_arg2, B, N1, N2, D, mode, grad_preds);
  HG_CHECK_LAUNCH("set_loss_bwd_kernel(preds)");
  if (grad_gts) {
    HgCsr rev1;
    rev1.off = nullptr;
    rev1.list = nullptr;
    if (g1) {
      rc = hg_csr_build_unordered(arg1, B, N1, N2, w.rev1.ptr, w.rev1.bytes, &rev1, stream);
      if (rc) return rc;
    }
    const long long tg = (long long)B * N2 * (D > 8 ? D : 1);
    set_loss_bwd_kernel<<<hg_grid_for(tg, 256, 16), 256, 0, stream>>>(gts, preds, arg2, rev1.off, rev1.list, arg1, g2, g1,
                                                                      hd_arg2, hd_arg1, B, N2, N1, D, mode, grad_gts);
    HG_CHECK_LAUNCH("set_loss_bwd_kernel(gts)");
  }
  return HG_OK;
}
