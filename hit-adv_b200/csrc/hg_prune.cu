// hg_prune.cu -- exact, spatially pruned nearest-neighbour (Chamfer, both directions) and self-kNN passes for large
// clouds.
//
// The all-pairs kernels (hg_nn_bidir.cu, hg_knn3.cu) evaluate every (query, candidate) pair; at 16384 points a query's
// few nearest neighbours lie within ~1 % of the cloud.  Here every cloud is first put in kd-tree order (leaves of 32
// points with tight axis-aligned boxes), then a warp owns one leaf of 32 queries and visits candidate leaves in
// tree order starting from the nearest one (own leaf for self-kNN), skipping a whole leaf when no lane can find
// anything in it:
//     lowerbound(D^2(query or query box, leaf box)) > thr + slack,    slack = 1.5e-6 (S + thr) >= 24 u (S + thr),
// D^2 computed with rounding toward -inf, thr the lane's current exact threshold (1-NN: best value so far; kNN: the
// k-th listed value nudged up one ulp, or a seed), S = (|q| + max|c|)^2.  The reference's FP32 value undershoots the
// real squared distance by at most ~9 u S (DESIGN 5.1, 5.2), so a skipped leaf holds no candidate whose reference
// value is <= thr: ties at the threshold are always visited.  Visited leaves go through the packed arithmetic of the
// all-pairs kernels (Chamfer: P = (rx + ry) + zz', zz' = fma(x2',y2, fma(x1',y1, x0'*y0)), x' = -2x, which gives the
// same bits with the roles of the two points swapped; kNN: the 4-operation folded sign-bit filter and an exact drain).
// Leaves are not visited in index order, so every selection compares (value, original index) lexicographically:
// results equal the all-pairs kernels' bit for bit (first index among equal values).
//
// A cloud with a non-finite coordinate or a squared norm >= 1e36 is flagged by the ordering build; the search skips
// it and the caller runs the all-pairs kernels on the flagged clouds only (documented NaN behaviour unchanged).
#include <string.h>

#include "hg_common.cuh"

namespace {

constexpr int kLeaf = 32;
constexpr int kIdxBits = 14;  // sort keys: 18 bits of quantised coordinate, 14 bits of point index
constexpr unsigned kIdxMask = (1u << kIdxBits) - 1u;
constexpr unsigned kPadKey = 0xffffffffu;
constexpr float kQuantMax = 262142.f;  // 2^18 - 2: a real key never equals kPadKey
constexpr int kBuildThreads = 1024;
constexpr int kSearchWarps = 4;
constexpr float kSlack = 1.5e-6f;  // >= 24 u, u = 2^-24

// nn: visited, total leaf pairs; knn: visited, total, then drains, candidates inserted, warp rounds of the drains
__device__ unsigned long long g_prune_tiles[7];

__device__ __forceinline__ float gap_rd(float alo, float ahi, float blo, float bhi) {
  return fmaxf(fmaxf(__fsub_rd(blo, ahi), __fsub_rd(alo, bhi)), 0.f);
}
// lower bound on the squared distance between two boxes (a point is a box with lo == hi)
__device__ __forceinline__ float box_d2_rd(float4 alo, float4 ahi, float4 blo, float4 bhi) {
  const float gx = gap_rd(alo.x, ahi.x, blo.x, bhi.x), gy = gap_rd(alo.y, ahi.y, blo.y, bhi.y),
              gz = gap_rd(alo.z, ahi.z, blo.z, bhi.z);
  return __fadd_rd(__fadd_rd(__fmul_rd(gx, gx), __fmul_rd(gy, gy)), __fmul_rd(gz, gz));
}
__device__ __forceinline__ bool may_hold(float lb, float thr, float S) { return !(lb > thr + kSlack * (S + thr)); }

__device__ unsigned long long g_order_counts[3];  // orderings: refit and kept, rebuilt from a state, built without one

// Leaf L's box from the warp's 32 points (v, real when `in`), written to o.box; returns h + the leaf's
// (ext_x + ext_y + ext_z), accumulated on lane 0.  The build and the refit both go through here, so H_built and the
// refit's H are the same bits for the same permutation and points.
__device__ __forceinline__ float leaf_box(const HgPruneOrder &o, int b, int nleaf, int L, int lane, bool in,
                                          const float (&v)[3], float h) {
  float lo[3], hi[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    lo[c] = hg_warp_min_f32(in ? v[c] : CUDART_INF_F);
    hi[c] = hg_warp_max_f32(in ? v[c] : -CUDART_INF_F);
  }
  if (lane == 0) {
    o.box[((size_t)b * nleaf + L) * 2] = make_float4(lo[0], lo[1], lo[2], 0.f);
    o.box[((size_t)b * nleaf + L) * 2 + 1] = make_float4(hi[0], hi[1], hi[2], 0.f);
    h += ((hi[0] - lo[0]) + (hi[1] - lo[1])) + (hi[2] - lo[2]);
  }
  return h;
}
// sum of the per-warp leaf sums (lane 0 of every warp) in warp order; the result is valid on thread 0
__device__ __forceinline__ float block_sum_leaves(float h, float *s_h) {
  const int tid = threadIdx.x;
  if ((tid & 31) == 0) s_h[tid >> 5] = h;
  __syncthreads();
  float H = 0.f;
  if (tid == 0)
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) H += s_h[w];
  return H;
}

// ---- ordering build: one CTA per cloud, kd splits (median of the longest axis) by selection -----------------------
// The tree: the positions [0, Np) (Np = N padded to a power of two, padding at positions >= N) are split level by level
// into segments of s = Np, Np/2, ..., 64 entries.  A segment's key of a point is (quantised coordinate on the
// segment's longest axis) << 14 | point index, so keys are distinct, and the left child of a segment is exactly its
// s/2 smallest keys (all of its real points when it holds s/2 or fewer; padding sorts after every real key).  The box,
// the axis, the scale and so the next level's keys depend only on which points a segment holds, so the order of the
// points inside a segment matters only at the last level, where each 64-entry segment is sorted by its key and that
// order is the permutation.  Correctness never depends on the quality of a split: the leaf boxes are recomputed from
// the points.
//
// Warp w of the first nw = Np / (32 E) warps holds the positions [w 32E, (w + 1) 32E), entry (h, lane) at w 32E + 32h +
// lane.  Levels whose segments span several warps run CTA-wide: the segment's rank-(s/2 - 1) key by an MSD radix
// select (8-bit digits, a shared-memory histogram per segment, one warp per segment scans it), then one in-place
// partition (ballots and popc within a warp, the counts of the segment's earlier warps).  From 32E entries down, a
// warp finishes its own entries in registers: per level, each group's box from warp reductions, its keys, and a
// bitonic sort of the group with shuffles (the last one is the 64-entry sort that fixes the leaf order).
//
// With an ordering state (hdr != null: o.perm points into the state, hdr is its per-cloud header) the kernel runs after
// prune_refit_kernel and rebuilds only the clouds the refit marked (info.z != 0); it then also stores the leaf-box
// quality H of the new permutation in the header.  count (null, or g_order_counts): clouds ordered without a state.
constexpr int kCtaSegs = kBuildThreads / 32 / 2;  // segments of the CTA-wide levels: at most half the warps

struct SegSplit {
  int ax;
  float lo, scale;
};
// split of a segment from its box (ordered-int min / max per coordinate): the axis of the largest extent (strict >),
// its low end and the quantisation scale
__device__ __forceinline__ SegSplit seg_split(const unsigned (&mn)[3], const unsigned (&mx)[3]) {
  SegSplit sp = {0, hg_unord(mn[0]), 0.f};
  float ext = hg_unord(mx[0]) - sp.lo;
#pragma unroll
  for (int c = 1; c < 3; ++c) {
    const float lo = hg_unord(mn[c]), e = hg_unord(mx[c]) - lo;
    if (e > ext) {
      sp.ax = c;
      sp.lo = lo;
      ext = e;
    }
  }
  sp.scale = ext > 0.f ? kQuantMax / ext : 0.f;
  return sp;
}
__device__ __forceinline__ unsigned split_key(const float *p, unsigned id, SegSplit sp) {
  const float f = (p[(size_t)id * 3 + sp.ax] - sp.lo) * sp.scale;
  return ((unsigned)fminf(fmaxf(f, 0.f), kQuantMax) << kIdxBits) | id;
}
__device__ __forceinline__ void box_add(const float *p, unsigned id, unsigned (&mn)[3], unsigned (&mx)[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const unsigned u = hg_ord(p[(size_t)id * 3 + c]);
    mn[c] = min(mn[c], u);
    mx[c] = max(mx[c], u);
  }
}

// Ascending bitonic sort of every group of G consecutive register rows (32 G entries, entry (h, lane) is element
// 32 (h % G) + lane of group h / G), in registers with shuffles.
template <int E, int G>
__device__ __forceinline__ void warp_sort_groups(unsigned (&k)[E], int lane) {
#pragma unroll
  for (int kk = 2; kk <= 32 * G; kk <<= 1) {
#pragma unroll
    for (int j = kk >> 1; j > 0; j >>= 1) {
      if (j >= 32) {
        const int jh = j >> 5;
#pragma unroll
        for (int h = 0; h < E; ++h) {
          if ((h & jh) == 0) {
            const bool asc = (((h % G) << 5) & kk) == 0;
            const unsigned lo = min(k[h], k[h | jh]), hi = max(k[h], k[h | jh]);
            k[h] = asc ? lo : hi;
            k[h | jh] = asc ? hi : lo;
          }
        }
      } else {
        const bool lower = (lane & j) == 0;
#pragma unroll
        for (int h = 0; h < E; ++h) {
          const unsigned y = __shfl_xor_sync(0xffffffffu, k[h], j);
          const bool asc = ((((h % G) << 5) | lane) & kk) == 0;
          k[h] = lower == asc ? min(k[h], y) : max(k[h], y);
        }
      }
    }
  }
}

// The warp-local levels from groups of G rows down to 2 rows (64 entries): per group of 32 G entries the box (padding
// is kPadKey), the keys, then the sort of every group.
template <int E, int G>
__device__ __forceinline__ void warp_levels(const float *p, unsigned (&v)[E], int lane) {
#pragma unroll
  for (int g = 0; g < E; g += G) {
    unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
#pragma unroll
    for (int h = g; h < g + G; ++h)
      if (v[h] != kPadKey) box_add(p, v[h] & kIdxMask, lo, hi);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      lo[c] = __reduce_min_sync(0xffffffffu, lo[c]);
      hi[c] = __reduce_max_sync(0xffffffffu, hi[c]);
    }
    const SegSplit sp = seg_split(lo, hi);
#pragma unroll
    for (int h = g; h < g + G; ++h)
      if (v[h] != kPadKey) v[h] = split_key(p, v[h] & kIdxMask, sp);
  }
  warp_sort_groups<E, G>(v, lane);
  if constexpr (G > 2) warp_levels<E, G / 2>(p, v, lane);
}

// E = entries per lane (Np / 1024 from 2048 points up, else 2)
template <bool CHAMFER_NORM, int E>
__global__ void __launch_bounds__(kBuildThreads, 1) prune_order_kernel(const float *__restrict__ pc, int N, int Np,
                                                                       HgPruneOrder o, float4 *hdr,
                                                                       unsigned long long *count) {
  extern __shared__ unsigned sid[];  // [Np] point indices in tree order
  __shared__ unsigned smin[3][kCtaSegs], smax[3][kCtaSegs];
  __shared__ SegSplit ssplit[kCtaSegs];
  __shared__ unsigned hist[kCtaSegs][256], spref[kCtaSegs], srank[kCtaSegs], swl[kBuildThreads / 32];
  __shared__ unsigned s_bad, s_norm;
  __shared__ float s_h[kBuildThreads / 32];
  constexpr int C = 32 * E;  // entries per warp
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (hdr != nullptr && o.info[b].z == 0.f) return;  // the refit kept this cloud's ordering
  if (count != nullptr && hdr == nullptr && tid == 0) atomicAdd(count + 2, 1ull);
  const float *p = pc + (size_t)b * N * 3;
  if (tid == 0) {
    s_bad = 0u;
    s_norm = 0u;
  }
  for (int t = tid; t < kCtaSegs * 256; t += kBuildThreads) (&hist[0][0])[t] = 0u;
  __syncthreads();
  float mn = 0.f;
  bool bad = false;
  for (int i = tid; i < N; i += kBuildThreads) {
    sid[i] = (unsigned)i;
    const float x = p[(size_t)i * 3], y = p[(size_t)i * 3 + 1], z = p[(size_t)i * 3 + 2];
    bad |= !(isfinite(x) && isfinite(y) && isfinite(z));
    mn = fmaxf(mn, fmaf(z, z, fmaf(y, y, x * x)));
  }
  mn = hg_warp_max_f32(mn);
  bad = __any_sync(0xffffffffu, bad);
  if (lane == 0) {
    atomicMax(&s_norm, __float_as_uint(mn));
    if (bad) s_bad = 1u;
  }
  __syncthreads();
  const float norm = __uint_as_float(s_norm);
  const bool flagged = s_bad != 0u || !(norm < 1e36f);
  if (tid == 0) o.info[b] = make_float4(norm * 1.0001f, flagged ? 1.f : 0.f, 0.f, 0.f);
  if (flagged) return;

  const bool active = warp < Np / C;
  const int wbase = warp * C;
  unsigned v[E];  // the warp's entries: point indices, then this level's keys
  // CTA-wide levels: segments of 2C .. Np entries
  for (int s = Np; s > C; s >>= 1) {
    const int nseg = Np / s, seg = wbase / s, sbase = seg * s;
    if (tid < nseg)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        smin[c][tid] = 0xffffffffu;
        smax[c][tid] = 0u;
      }
    __syncthreads();
    if (active) {
      unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
#pragma unroll
      for (int h = 0; h < E; ++h) {
        const int pos = wbase + 32 * h + lane;
        if (pos < N) {
          v[h] = sid[pos];
          box_add(p, v[h], lo, hi);
        }
      }
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        lo[c] = __reduce_min_sync(0xffffffffu, lo[c]);
        hi[c] = __reduce_max_sync(0xffffffffu, hi[c]);
        if (lane == 0) {
          atomicMin(&smin[c][seg], lo[c]);
          atomicMax(&smax[c][seg], hi[c]);
        }
      }
    }
    __syncthreads();
    if (tid < nseg) {
      unsigned lo[3], hi[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        lo[c] = smin[c][tid];
        hi[c] = smax[c][tid];
      }
      ssplit[tid] = seg_split(lo, hi);
      spref[tid] = 0u;
      srank[tid] = s / 2 - 1;
    }
    __syncthreads();
    // a segment with s/2 real points or fewer keeps them where they are (all in its left half)
    const bool split = active && N - sbase > s / 2;
    if (split) {
      const SegSplit sp = ssplit[seg];
#pragma unroll
      for (int h = 0; h < E; ++h)
        if (wbase + 32 * h + lane < N) v[h] = split_key(p, v[h], sp);
    }
    for (int shift = 24; shift >= 0; shift -= 8) {  // radix select of the rank-(s/2 - 1) key
      if (split) {
        const unsigned pref = spref[seg], hmask = shift == 24 ? 0u : 0xffffffffu << (shift + 8);
#pragma unroll
        for (int h = 0; h < E; ++h)
          if (wbase + 32 * h + lane < N && ((v[h] ^ pref) & hmask) == 0u)
            atomicAdd(&hist[seg][(v[h] >> shift) & 255u], 1u);
      }
      __syncthreads();
      if (warp < nseg && N - warp * s > s / 2) {  // warp `warp` finds the digit of segment `warp`, clears its bins
        const unsigned r = srank[warp];
        unsigned cnt[8], loc = 0u;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          cnt[i] = hist[warp][lane * 8 + i];
          hist[warp][lane * 8 + i] = 0u;
          loc += cnt[i];
        }
        unsigned inc = loc;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const unsigned t = __shfl_up_sync(0xffffffffu, inc, d);
          if (lane >= d) inc += t;
        }
        unsigned acc = inc - loc;
        if (acc <= r && r < inc) {
          bool found = false;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            if (!found && r < acc + cnt[i]) {
              found = true;
              spref[warp] |= (unsigned)(lane * 8 + i) << shift;
              srank[warp] = r - acc;
            }
            acc += cnt[i];
          }
        }
      }
      __syncthreads();
    }
    // partition: keys <= the selected one to the left half, the others after it
    const unsigned m = split ? spref[seg] : 0u;
    if (split) {
      unsigned nl = 0u;
#pragma unroll
      for (int h = 0; h < E; ++h) nl += __popc(__ballot_sync(0xffffffffu, wbase + 32 * h + lane < N && v[h] <= m));
      if (lane == 0) swl[warp] = nl;
    }
    __syncthreads();
    if (split) {
      unsigned before = 0u;  // left keys of the segment's earlier warps, then of earlier entries
      for (int w = sbase / C; w < warp; ++w) before += swl[w];
#pragma unroll
      for (int h = 0; h < E; ++h) {
        const int pos = wbase + 32 * h + lane;
        const bool real = pos < N, left = real && v[h] <= m;
        const unsigned bal = __ballot_sync(0xffffffffu, left);
        const int lb = (int)(before + __popc(bal & ((1u << lane) - 1u)));
        if (real) sid[left ? sbase + lb : sbase + s / 2 + (pos - sbase - lb)] = v[h] & kIdxMask;
        before += __popc(bal);
      }
    }
    __syncthreads();
  }
  // warp-local levels: groups of G rows (32 G entries), G = E .. 2
  if (active) {
#pragma unroll
    for (int h = 0; h < E; ++h) {
      const int pos = wbase + 32 * h + lane;
      v[h] = pos < N ? sid[pos] : kPadKey;
    }
    warp_levels<E, E>(p, v, lane);
#pragma unroll
    for (int h = 0; h < E; ++h) sid[wbase + 32 * h + lane] = v[h] & kIdxMask;
  }
  __syncthreads();

  for (int i = tid; i < N; i += kBuildThreads) {
    const int id = (int)sid[i];
    const float x = p[(size_t)id * 3], y = p[(size_t)id * 3 + 1], z = p[(size_t)id * 3 + 2];
    const float w = CHAMFER_NORM ? hg_dot3_fma(x, y, z, x, y, z) : hg_sumsq3_seq(x, y, z);
    o.pts[(size_t)b * N + i] = make_float4(x, y, z, w);
    o.perm[(size_t)b * N + i] = id;
  }
  const int nleaf = (N + kLeaf - 1) / kLeaf;
  float h = 0.f;
  for (int L = tid >> 5; L < nleaf; L += kBuildThreads / 32) {
    const int i = L * kLeaf + lane;
    float v[3] = {0.f, 0.f, 0.f};
    if (i < N) {
      const int id = (int)sid[i];
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = p[(size_t)id * 3 + c];
    }
    h = leaf_box(o, b, nleaf, L, lane, i < N, v, h);
  }
  if (hdr != nullptr) {
    const float H = block_sum_leaves(h, s_h);
    if (tid == 0) hdr[b] = make_float4(H, 0.f, 0.f, 0.f);
  }
}

// ---- ordering state: refit of the previous call's permutation ---------------------------------------------------------
// One CTA per cloud.  Validates the state's permutation (every entry in [0, N), each index once: a bitmap in shared
// memory), recomputes the per-cloud info exactly as the build does (the max and the any-non-finite test do not depend
// on the order), gathers the points through the permutation (pts in the form's norm arithmetic and leaf boxes, bit for
// bit what prune_order_kernel writes for the same permutation) and measures H = sum over leaves of the box's
// (ext_x + ext_y + ext_z).  The cloud is marked for the rebuild (info.z = 1) when the permutation is invalid or
// !(H <= (1 + tol) H_built): a NaN or garbage header fails the comparison too.  STAGE: the cloud is staged in shared
// memory (12 B per point) for the gather instead of being read again from global memory (L2).
template <bool CHAMFER_NORM, bool STAGE>
__global__ void __launch_bounds__(kBuildThreads) prune_refit_kernel(const float *__restrict__ pc, int N, HgPruneOrder o,
                                                                    const float4 *__restrict__ hdr, float tol,
                                                                    unsigned long long *count) {
  extern __shared__ float spts[];  // STAGE: [N * 3]
  __shared__ unsigned bits[HG_PRUNE_MAX_N / 32];
  __shared__ unsigned s_bad, s_norm, s_invalid;
  __shared__ float s_h[kBuildThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  const float *p = pc + (size_t)b * N * 3;
  const int *perm = o.perm + (size_t)b * N;
  for (int t = tid; t < (N + 31) / 32; t += kBuildThreads) bits[t] = 0u;
  if (tid == 0) {
    s_bad = 0u;
    s_norm = 0u;
    s_invalid = 0u;
  }
  __syncthreads();
  float mn = 0.f;
  bool bad = false, invalid = false;
  for (int i = tid; i < N; i += kBuildThreads) {
    const float x = p[(size_t)i * 3], y = p[(size_t)i * 3 + 1], z = p[(size_t)i * 3 + 2];
    bad |= !(isfinite(x) && isfinite(y) && isfinite(z));
    mn = fmaxf(mn, fmaf(z, z, fmaf(y, y, x * x)));
    if (STAGE) {
      spts[i * 3] = x;
      spts[i * 3 + 1] = y;
      spts[i * 3 + 2] = z;
    }
    const int id = perm[i];
    if ((unsigned)id >= (unsigned)N) {
      invalid = true;
    } else {
      const unsigned bit = 1u << (id & 31);
      invalid |= (atomicOr(&bits[id >> 5], bit) & bit) != 0u;  // N entries in range, none twice: a permutation
    }
  }
  mn = hg_warp_max_f32(mn);
  bad = __any_sync(0xffffffffu, bad);
  invalid = __any_sync(0xffffffffu, invalid);
  if (lane == 0) {
    atomicMax(&s_norm, __float_as_uint(mn));
    if (bad) s_bad = 1u;
    if (invalid) s_invalid = 1u;
  }
  __syncthreads();
  const float norm = __uint_as_float(s_norm);
  const bool flagged = s_bad != 0u || !(norm < 1e36f);
  if (flagged || s_invalid != 0u) {  // flagged: the all-pairs kernels take the cloud, nothing else to write
    if (tid == 0) {
      o.info[b] = make_float4(norm * 1.0001f, flagged ? 1.f : 0.f, flagged ? 0.f : 1.f, 0.f);
      if (count != nullptr) atomicAdd(count + (flagged ? 0 : 1), 1ull);
    }
    return;
  }
  const int nleaf = (N + kLeaf - 1) / kLeaf;
  float h = 0.f;
  for (int L = tid >> 5; L < nleaf; L += kBuildThreads / 32) {  // the build's thread-to-point map, one pass
    const int i = L * kLeaf + lane;
    float v[3] = {0.f, 0.f, 0.f};
    if (i < N) {
      const int id = perm[i];
#pragma unroll
      for (int c = 0; c < 3; ++c) v[c] = STAGE ? spts[id * 3 + c] : p[(size_t)id * 3 + c];
      const float w = CHAMFER_NORM ? hg_dot3_fma(v[0], v[1], v[2], v[0], v[1], v[2]) : hg_sumsq3_seq(v[0], v[1], v[2]);
      o.pts[(size_t)b * N + i] = make_float4(v[0], v[1], v[2], w);
    }
    h = leaf_box(o, b, nleaf, L, lane, i < N, v, h);
  }
  const float H = block_sum_leaves(h, s_h);
  if (tid == 0) {
    const bool rebuild = !(H <= (1.f + tol) * hdr[b].x);
    o.info[b] = make_float4(norm * 1.0001f, 0.f, rebuild ? 1.f : 0.f, 0.f);
    if (count != nullptr) atomicAdd(count + (rebuild ? 1 : 0), 1ull);
  }
}

struct PruneSearch {
  HgPruneOrder q, c;
  int self;  // candidates are the query cloud (self-kNN): the visit starts at the query's own leaf
  int k1;
  float *vals;        // kNN [B,Nq,k1] (may be null), 1-NN [B,Nq]
  int *idx;           // same shape
  int *idx_state;     // kNN: second copy of idx or null
  const float *thr0;  // kNN: [B,Nq] exact upper bounds by original index, or null
  unsigned long long *count;  // null, or {visited leaf pairs, all leaf pairs} (kNN: then the three drain counts)
};

// List of the k1 smallest (value, index) pairs in lexicographic order, ascending, held in registers and indexed only
// by constants.  The k1 live entries are the tail [KM - k1, KM); the head holds (-inf, -1), which no candidate sorts
// before, so the k1-th value is always v[KM - 1].
template <int KM>
struct LexTopK {
  float v[KM];
  int id[KM];
  __device__ __forceinline__ void init(int k1) {
#pragma unroll
    for (int t = 0; t < KM; ++t) {
      v[t] = t < KM - k1 ? -CUDART_INF_F : CUDART_INF_F;
      id[t] = t < KM - k1 ? -1 : 0;
    }
  }
  __device__ __forceinline__ bool sorts_before(float d, int j, int t) const {
    return (d < v[t]) | ((d == v[t]) & (j < id[t]));  // no short-circuit: no branch
  }
  // Insertion as one pass of predicated compare-exchange steps: entry t takes entry t - 1 when (d, j) sorts before
  // that, else (d, j) when it sorts before entry t.  (+inf, INT_MAX) sorts before nothing: a no-op.
  __device__ __forceinline__ void push(float d, int j) {
    bool before = sorts_before(d, j, KM - 1);
#pragma unroll
    for (int t = KM - 1; t > 0; --t) {
      const bool prev = sorts_before(d, j, t - 1);
      v[t] = prev ? v[t - 1] : before ? d : v[t];
      id[t] = prev ? id[t - 1] : before ? j : id[t];
      before = prev;
    }
    v[0] = before ? d : v[0];
    id[0] = before ? j : id[0];
  }
};

// not hg_nudge_up, which maps NaN to +inf: with that form prune_search_kernel compiles to different machine code
__device__ __forceinline__ float nudge_up(float v) { return v < CUDART_INF_F ? nextafterf(v, CUDART_INF_F) : v; }

// Resident CTAs per SM the search's register allocation must allow (0: no bound).  KM = 20: 4, since without a bound
// ptxas stops at 96 registers and spills.  KM = 6 stays unbounded (72 registers, 7 CTAs): a bound of 8 CTAs
// (64 registers) measured slower, 8.91 against 8.79 ms per 1024 x 16384 call (DESIGN 5.5).
template <int KM>
constexpr int kSearchMinCtas = KM == 20 ? 4 : 0;

// KM == 1: 1-NN with the Chamfer arithmetic; KM > 1: kNN list with the KNNDist arithmetic and the folded filter.
template <int KM>
__global__ void __launch_bounds__(kSearchWarps * 32, kSearchMinCtas<KM>) prune_search_kernel(PruneSearch a) {
  __shared__ float4 tile[kSearchWarps][kLeaf];  // 16 candidate pairs: (c0_j,c0_j1,c1_j,c1_j1), (c2_j,c2_j1,w_j,w_j1)
  __shared__ int tperm[kSearchWarps][kLeaf];
  constexpr bool kNN1 = KM == 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, b = blockIdx.y;
  const int Nq = a.q.N, Nc = a.c.N;
  const int nlq = (Nq + kLeaf - 1) / kLeaf, nlc = (Nc + kLeaf - 1) / kLeaf;
  const int Lq = blockIdx.x * kSearchWarps + warp;
  if (Lq >= nlq) return;
  const float4 qinfo = a.q.info[b], cinfo = a.c.info[b];
  if (qinfo.y != 0.f || cinfo.y != 0.f) return;  // all-pairs kernels take this cloud

  const int pos = Lq * kLeaf + lane;
  const bool valid = pos < Nq;
  const float4 qp = valid ? a.q.pts[(size_t)b * Nq + pos] : make_float4(0.f, 0.f, 0.f, 0.f);
  const int qid = valid ? a.q.perm[(size_t)b * Nq + pos] : 0;
  const float a0 = -2.0f * qp.x, a1 = -2.0f * qp.y, a2 = -2.0f * qp.z, rq = qp.w;
  const float cmax = sqrtf(cinfo.x);
  const float S = (sqrtf(rq) + cmax) * (sqrtf(rq) + cmax) * 1.0001f;
  const float Sw = hg_warp_max_f32(valid ? S : 0.f);
  const float4 *qbox = a.q.box + (size_t)b * nlq * 2;
  const float4 *cbox = a.c.box + (size_t)b * nlc * 2;
  const float4 *cpts = a.c.pts + (size_t)b * Nc;
  const int *cperm = a.c.perm + (size_t)b * Nc;
  const float4 qlo = qbox[2 * Lq], qhi = qbox[2 * Lq + 1];
  const float4 qpt = make_float4(qp.x, qp.y, qp.z, 0.f);
  float *tf = reinterpret_cast<float *>(tile[warp]);

  auto stage = [&](int L) {
    const int cpos = L * kLeaf + lane;
    const float4 c = cpos < Nc ? cpts[cpos] : make_float4(0.f, 0.f, 0.f, CUDART_INF_F);
    const int cid = cpos < Nc ? cperm[cpos] : 0x7fffffff;
    __syncwarp();
    const int pp = lane >> 1, h = lane & 1;
    tf[8 * pp + h] = c.x;
    tf[8 * pp + 2 + h] = c.y;
    tf[8 * pp + 4 + h] = c.z;
    tf[8 * pp + 6 + h] = c.w;
    tperm[warp][lane] = cid;
    __syncwarp();
  };

  // first leaf: the query's own (self) or the one whose centre is nearest to the query leaf's centre
  int Ls = Lq;
  if (!a.self) {
    float bd = CUDART_INF_F;
    int bi = 0;
    const float cx = 0.5f * (qlo.x + qhi.x), cy = 0.5f * (qlo.y + qhi.y), cz = 0.5f * (qlo.z + qhi.z);
    for (int L = lane; L < nlc; L += 32) {
      const float4 lo = cbox[2 * L], hi = cbox[2 * L + 1];
      const float dx = 0.5f * (lo.x + hi.x) - cx, dy = 0.5f * (lo.y + hi.y) - cy, dz = 0.5f * (lo.z + hi.z) - cz;
      const float d = dx * dx + dy * dy + dz * dz;
      if (d < bd) {
        bd = d;
        bi = L;
      }
    }
    const float wm = hg_warp_min_f32(bd);
    Ls = __reduce_min_sync(0xffffffffu, bd == wm ? bi : 0x7fffffff);
    if (Ls == 0x7fffffff) Ls = 0;
  }

  float best = CUDART_INF_F;  // 1-NN
  int bid = 0x7fffffff;
  LexTopK<kNN1 ? 1 : KM> top;
  float seed = CUDART_INF_F, thr = CUDART_INF_F;
  unsigned ndrain = 0u, nround = 0u, npush = 0u;  // kNN drains, warp-uniform; npush per lane
  // exact values of the staged candidates in `sub` inserted into the list, all lanes in lockstep: a lane whose
  // candidates are done inserts (+inf, INT_MAX)
  auto drain = [&](unsigned sub) {
    ++ndrain;
    while (__any_sync(0xffffffffu, sub != 0u)) {
      const int c = (__ffs(sub) - 1) & (kLeaf - 1);
      const bool take = sub != 0u;
      sub &= sub - 1u;
      const int pp = c >> 1, h = c & 1;
      const float c0 = tf[8 * pp + h], c1 = tf[8 * pp + 2 + h], c2 = tf[8 * pp + 4 + h], cw = tf[8 * pp + 6 + h];
      // knn_dist_exact<EXPANDED>: (xx_j + nzz) + xx_i
      const float d = __fadd_rn(__fadd_rn(cw, __fmaf_rn(a2, c2, __fmaf_rn(a1, c1, __fmul_rn(a0, c0)))), rq);
      const int j = tperm[warp][c];
      top.push(take ? d : CUDART_INF_F, take ? j : 0x7fffffff);
      ++nround;
      npush += take ? 1u : 0u;
    }
  };
  int dfirst = 0;  // the first leaf Ls ^ d the main loop visits
  unsigned long long visited = 0;
  if (!kNN1) {
    top.init(a.k1);
    if (a.thr0 != nullptr) {
      seed = valid ? a.thr0[(size_t)b * Nq + qid] : CUDART_INF_F;
    } else if (KM <= kLeaf) {
      // seed: the k1-th smallest exact distance over the own leaf (real candidates: an exact upper bound), from a
      // value-only min/max network over the list's layout
      stage(Ls);
      for (int c = 0; c < kLeaf; ++c) {
        const int pp = c >> 1, h = c & 1;
        const float c0 = tf[8 * pp + h], c1 = tf[8 * pp + 2 + h], c2 = tf[8 * pp + 4 + h], cw = tf[8 * pp + 6 + h];
        hg_sorted_min_insert(top.v, __fadd_rn(__fadd_rn(cw, __fmaf_rn(a2, c2, __fmaf_rn(a1, c1, __fmul_rn(a0, c0)))), rq));
      }
      const float kth = top.v[KM - 1];
      seed = valid ? nudge_up(kth) : CUDART_INF_F;
      // the own leaf's visit: its candidates at or below the k1-th value fill the list, which leaves the threshold
      // at the seed; the main loop starts at its sibling
      top.init(a.k1);
      unsigned sub = 0u;
      for (int c = 0; c < kLeaf; ++c) {
        const int pp = c >> 1, h = c & 1;
        const float c0 = tf[8 * pp + h], c1 = tf[8 * pp + 2 + h], c2 = tf[8 * pp + 4 + h], cw = tf[8 * pp + 6 + h];
        const float d = __fadd_rn(__fadd_rn(cw, __fmaf_rn(a2, c2, __fmaf_rn(a1, c1, __fmul_rn(a0, c0)))), rq);
        sub |= (valid && d <= kth ? 1u : 0u) << c;
      }
      drain(sub);
      visited = 1;
      dfirst = 1;
    }
    thr = seed;
  }
  if (!valid) thr = -CUDART_INF_F;  // padding lanes never need a leaf

  int P2 = 1;
  while (P2 < nlc) P2 <<= 1;
  for (int d0 = 0; d0 < P2; d0 += 32) {
    // warp-uniform test of 32 leaves against the largest current threshold of the warp, box against box
    const float tw = hg_warp_max_f32(thr);
    const int Lt = Ls ^ (d0 + lane);
    bool pass = false;
    if (Lt < nlc && d0 + lane >= dfirst) pass = may_hold(box_d2_rd(qlo, qhi, cbox[2 * Lt], cbox[2 * Lt + 1]), tw, Sw);
    unsigned m = __ballot_sync(0xffffffffu, pass);
    while (m) {
      const int bit = __ffs(m) - 1;
      m &= m - 1u;
      const int L = Ls ^ (d0 + bit);
      // re-test against every lane's current threshold, point against box
      const float4 clo = cbox[2 * L], chi = cbox[2 * L + 1];
      const bool need = may_hold(box_d2_rd(qpt, qpt, clo, chi), thr, S);
      if (!__any_sync(0xffffffffu, need)) continue;
      ++visited;
      stage(L);
      if (kNN1) {
        float mv = CUDART_INF_F;
#pragma unroll 4
        for (int pp = 0; pp < kLeaf / 2; ++pp) {
          const float4 A = tile[warp][2 * pp], Bv = tile[warp][2 * pp + 1];
          float2 t = __fmul2_rn(make_float2(a0, a0), make_float2(A.x, A.y));
          t = __ffma2_rn(make_float2(a1, a1), make_float2(A.z, A.w), t);
          t = __ffma2_rn(make_float2(a2, a2), make_float2(Bv.x, Bv.y), t);
          const float2 P = __fadd2_rn(__fadd2_rn(make_float2(rq, rq), make_float2(Bv.z, Bv.w)), t);
          mv = fminf(fminf(mv, P.x), P.y);
        }
        if (valid && mv <= best) {  // rare: find the first original index attaining mv in this leaf
          int id = 0x7fffffff;
          for (int c = 0; c < kLeaf; ++c) {
            const int pp = c >> 1, h = c & 1;
            const float c0 = tf[8 * pp + h], c1 = tf[8 * pp + 2 + h], c2 = tf[8 * pp + 4 + h], cw = tf[8 * pp + 6 + h];
            const float v = __fadd_rn(__fadd_rn(rq, cw), __fmaf_rn(a2, c2, __fmaf_rn(a1, c1, __fmul_rn(a0, c0))));
            if (v == mv) id = min(id, tperm[warp][c]);
          }
          if (mv < best || id < bid) {
            best = mv;
            bid = id;
          }
          thr = best;
        }
      } else {
        // folded 4-operation filter (hg_knn3.cu filter_addend / filter_value, FOLD4): sign bit = maybe below thr
        const float af = __fsub_rd(rq, __fadd_ru(thr, kSlack * (S + thr)));
        unsigned o = 0u;
#pragma unroll 4
        for (int pp = 0; pp < kLeaf / 2; ++pp) {
          const float4 A = tile[warp][2 * pp], Bv = tile[warp][2 * pp + 1];
          float2 t = __fadd2_rn(make_float2(Bv.z, Bv.w), make_float2(af, af));
          t = __ffma2_rn(make_float2(a2, a2), make_float2(Bv.x, Bv.y), t);
          t = __ffma2_rn(make_float2(a1, a1), make_float2(A.z, A.w), t);
          t = __ffma2_rn(make_float2(a0, a0), make_float2(A.x, A.y), t);
          o |= __float_as_uint(t.x) | __float_as_uint(t.y);
        }
        const bool hit = valid && (o >> 31) != 0u;
        if (__any_sync(0xffffffffu, hit)) {  // drain: which candidates, then exact values and insertion
          unsigned sub = 0u;
#pragma unroll 4
          for (int pp = 0; pp < kLeaf / 2; ++pp) {
            const float4 A = tile[warp][2 * pp], Bv = tile[warp][2 * pp + 1];
            float2 t = __fadd2_rn(make_float2(Bv.z, Bv.w), make_float2(af, af));
            t = __ffma2_rn(make_float2(a2, a2), make_float2(Bv.x, Bv.y), t);
            t = __ffma2_rn(make_float2(a1, a1), make_float2(A.z, A.w), t);
            t = __ffma2_rn(make_float2(a0, a0), make_float2(A.x, A.y), t);
            sub |= ((__float_as_uint(t.x) >> 31) << (2 * pp)) | ((__float_as_uint(t.y) >> 31) << (2 * pp + 1));
          }
          drain(hit ? sub : 0u);
          if (hit) thr = fminf(seed, nudge_up(top.v[KM - 1]));
        }
      }
    }
  }
  if (a.count != nullptr && lane == 0) {
    atomicAdd(a.count, visited);
    atomicAdd(a.count + 1, (unsigned long long)nlc);
  }
  if (!kNN1 && a.count != nullptr) {
    npush = __reduce_add_sync(0xffffffffu, npush);
    if (lane == 0) {
      atomicAdd(a.count + 2, (unsigned long long)ndrain);
      atomicAdd(a.count + 3, (unsigned long long)npush);
      atomicAdd(a.count + 4, (unsigned long long)nround);
    }
  }
  if (!valid) return;
  if (kNN1) {
    a.vals[(size_t)b * Nq + qid] = best;
    a.idx[(size_t)b * Nq + qid] = bid == 0x7fffffff ? 0 : bid;
  } else {
    const size_t o = ((size_t)b * Nq + qid) * a.k1;
#pragma unroll
    for (int t = 0; t < (kNN1 ? 1 : KM); ++t) {
      const int s = t - (KM - a.k1);  // the live entries are outputs 0 .. k1 - 1
      if (s >= 0) {
        if (a.vals) a.vals[o + s] = top.v[t];
        a.idx[o + s] = top.id[t];
        if (a.idx_state) a.idx_state[o + s] = top.id[t];
      }
    }
  }
}

template <int KM>
int launch_search(const PruneSearch &a, int B, cudaStream_t stream) {
  const int nlq = (a.q.N + kLeaf - 1) / kLeaf;
  dim3 grid((nlq + kSearchWarps - 1) / kSearchWarps, B);
  prune_search_kernel<KM><<<grid, kSearchWarps * 32, 0, stream>>>(a);
  HG_CHECK_LAUNCH("prune_search_kernel");
  return HG_OK;
}

int g_prune_mode = 1;     // hg_tune("prune", v): 0 = all-pairs kernels only, 1 = automatic
int g_prune_min_n = 0;    // hg_tune("prune_min_n", n): smallest cloud that takes the pruned path (0 = default)
int g_prune_count = 0;    // hg_tune("prune_count", 1): count visited leaf pairs and orderings (hg_prune_*counters)
int g_refit_tol = 0;      // hg_tune("prune_refit_tol", permille): rebuild threshold of the refit (0 = default)
int g_refit_stage = 0;    // hg_tune("prune_refit_stage", v): 0 = default, 1 = stage the cloud in shared memory, 2 = not

unsigned long long *counters() {
  if (!g_prune_count) return nullptr;
  void *ptr = nullptr;
  if (cudaGetSymbolAddress(&ptr, g_prune_tiles) != cudaSuccess) return nullptr;
  return (unsigned long long *)ptr;
}
unsigned long long *order_counters() {
  if (!g_prune_count) return nullptr;
  void *ptr = nullptr;
  if (cudaGetSymbolAddress(&ptr, g_order_counts) != cudaSuccess) return nullptr;
  return (unsigned long long *)ptr;
}

// an ordering in the workspace: points, permutation (unused with an ordering state), leaf boxes, per-cloud info
struct OrderLayout : HgPruneOrder {
  OrderLayout(HgCarve &c, int B, int N)
      : HgPruneOrder{c.take<float4>((size_t)B * N), c.take<int>((size_t)B * N),
                     c.take<float4>((size_t)B * ((N + kLeaf - 1) / kLeaf) * 2), c.take<float4>(B), N} {}
};

// an ordering state: the permutations, then the header (one float4 per cloud)
struct StateLayout {
  int *perm;
  float4 *hdr;
  StateLayout(HgCarve &c, int B, int N) : perm(c.take<int>((size_t)B * N)), hdr(c.take<float4>(B)) {}
};

}  // namespace

// Default size threshold: see DESIGN 5.1 / 5.2 (sweep with tools/prune_ab.py).
constexpr int kPruneDefaultMinN = 8192;
// Default refit tolerance tau [permille] and gather source: see DESIGN 5.5 (sweep with tools/order_state_ab.py).
constexpr int kRefitDefaultTolPermille = 100;
constexpr bool kRefitDefaultStage = true;

int hg_prune_tune(const char *key, int value) {
  if (!strcmp(key, "prune")) {
    g_prune_mode = value;
    return 1;
  }
  if (!strcmp(key, "prune_min_n")) {
    g_prune_min_n = value;
    return 1;
  }
  if (!strcmp(key, "prune_count")) {
    g_prune_count = value;
    return 1;
  }
  if (!strcmp(key, "prune_refit_tol")) {
    g_refit_tol = value;
    return 1;
  }
  if (!strcmp(key, "prune_refit_stage")) {
    g_refit_stage = value;
    return 1;
  }
  return 0;
}

bool hg_prune_applies(int N) {
  const int min_n = g_prune_min_n > 0 ? g_prune_min_n : kPruneDefaultMinN;
  return g_prune_mode != 0 && N >= min_n && N >= 2 * kLeaf && N <= HG_PRUNE_MAX_N;
}

size_t hg_prune_order_bytes(int B, int N) {
  if (B <= 0 || !hg_prune_applies(N)) return 0;
  return hg_layout_bytes<OrderLayout>(B, N);
}

HG_API size_t hg_order_state_bytes(int B, int N) {
  if (B <= 0 || N <= 0) return 0;
  return hg_layout_bytes<StateLayout>(B, N);
}

int hg_prune_build(const float *pc, int B, int N, bool chamfer_norm, void *ws, HgPruneOrder *o, cudaStream_t stream,
                   void *state) {
  *o = hg_layout_at<OrderLayout>(ws, B, N);
  const StateLayout s = hg_layout_at<StateLayout>(state, B, N);  // null pointers without a state
  float4 *hdr = s.hdr;
  if (state) o->perm = s.perm;  // with a state, the permutation lives there (the workspace slot is unused)
  int Np = 2 * kLeaf;
  while (Np < N) Np <<= 1;
  if (state) {
    const bool stage = g_refit_stage == 0 ? kRefitDefaultStage : g_refit_stage == 1;
    const float tol = (g_refit_tol > 0 ? g_refit_tol : kRefitDefaultTolPermille) * 1e-3f;
    const size_t rsmem = stage ? (size_t)N * 3 * sizeof(float) : 0;
    static HgPerDeviceOnce ronce[2];
    auto refit = chamfer_norm ? (stage ? prune_refit_kernel<true, true> : prune_refit_kernel<true, false>)
                              : (stage ? prune_refit_kernel<false, true> : prune_refit_kernel<false, false>);
    if (stage && ronce[chamfer_norm ? 1 : 0].first()) {
      HG_CUDA(cudaFuncSetAttribute(prune_refit_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   HG_PRUNE_MAX_N * 3 * (int)sizeof(float)));
      HG_CUDA(cudaFuncSetAttribute(prune_refit_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   HG_PRUNE_MAX_N * 3 * (int)sizeof(float)));
    }
    refit<<<B, kBuildThreads, rsmem, stream>>>(pc, N, *o, hdr, tol, order_counters());
    HG_CHECK_LAUNCH("prune_refit_kernel");
  }
  const size_t smem = (size_t)Np * sizeof(unsigned);
  static HgPerDeviceOnce once[2];
  // entries per lane: 32 warps of Np / 32 entries from 2048 points up, else Np / 64 warps of 64
  const int E = Np >= 32 * 64 ? Np / kBuildThreads : 2;
  auto pick = [](bool chamfer, int e) {
    if (chamfer) return e == 2 ? prune_order_kernel<true, 2> : e == 4 ? prune_order_kernel<true, 4>
                      : e == 8 ? prune_order_kernel<true, 8> : prune_order_kernel<true, 16>;
    return e == 2 ? prune_order_kernel<false, 2> : e == 4 ? prune_order_kernel<false, 4>
           : e == 8 ? prune_order_kernel<false, 8> : prune_order_kernel<false, 16>;
  };
  auto kernel = pick(chamfer_norm, E);
  if (once[chamfer_norm ? 1 : 0].first())
    for (int e = 2; e <= HG_PRUNE_MAX_N / kBuildThreads; e <<= 1)
      HG_CUDA(cudaFuncSetAttribute(pick(chamfer_norm, e), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   HG_PRUNE_MAX_N * (int)sizeof(unsigned)));
  // with a state: the clouds the refit marked only (the others exit at entry), so no host decision is needed
  kernel<<<B, kBuildThreads, smem, stream>>>(pc, N, Np, *o, hdr, order_counters());
  HG_CHECK_LAUNCH("prune_order_kernel");
  return HG_OK;
}

int hg_prune_nn_search(const HgPruneOrder &q, const HgPruneOrder &c, int B, float *mins, int *args,
                       cudaStream_t stream) {
  PruneSearch a;
  a.q = q;
  a.c = c;
  a.self = 0;
  a.k1 = 1;
  a.vals = mins;
  a.idx = args;
  a.idx_state = nullptr;
  a.thr0 = nullptr;
  a.count = counters();
  return launch_search<1>(a, B, stream);
}

int hg_prune_knn_search(const HgPruneOrder &o, int B, int k1, const float *thr0, float *vals, int *idx, int *idx_state,
                        cudaStream_t stream) {
  PruneSearch a;
  a.q = o;
  a.c = o;
  a.self = 1;
  a.k1 = k1;
  a.vals = vals;
  a.idx = idx;
  a.idx_state = idx_state;
  a.thr0 = thr0;
  a.count = counters();
  if (a.count) a.count += 2;
  if (k1 <= 6) return launch_search<6>(a, B, stream);
  if (k1 <= 20) return launch_search<20>(a, B, stream);
  if (k1 <= 32) return launch_search<32>(a, B, stream);
  return launch_search<64>(a, B, stream);
}

// Visited and total leaf pairs since the last call, {nn, nn total, knn, knn total}; synchronises the device.
HG_API int hg_prune_counters(unsigned long long *out4) {
  HG_REQUIRE(out4, HG_E_BADARG, "prune_counters: null pointer");
  HG_CUDA(cudaDeviceSynchronize());
  HG_CUDA(cudaMemcpyFromSymbol(out4, g_prune_tiles, sizeof(unsigned long long) * 4));
  const unsigned long long zero[4] = {0, 0, 0, 0};
  HG_CUDA(cudaMemcpyToSymbol(g_prune_tiles, zero, sizeof(zero)));
  return HG_OK;
}

// kNN drains since the last call, {drains, candidates inserted, warp rounds}; synchronises the device.
HG_API int hg_prune_drain_counters(unsigned long long *out3) {
  HG_REQUIRE(out3, HG_E_BADARG, "prune_drain_counters: null pointer");
  HG_CUDA(cudaDeviceSynchronize());
  HG_CUDA(cudaMemcpyFromSymbol(out3, g_prune_tiles, sizeof(unsigned long long) * 3, sizeof(unsigned long long) * 4));
  const unsigned long long zero[3] = {0, 0, 0};
  HG_CUDA(cudaMemcpyToSymbol(g_prune_tiles, zero, sizeof(zero), sizeof(unsigned long long) * 4));
  return HG_OK;
}

// Orderings since the last call, {refit and kept, rebuilt from a state, built without a state}, counted per cloud while
// hg_tune("prune_count", 1) is on; synchronises the device.
HG_API int hg_prune_order_counters(unsigned long long *out3) {
  HG_REQUIRE(out3, HG_E_BADARG, "prune_order_counters: null pointer");
  HG_CUDA(cudaDeviceSynchronize());
  HG_CUDA(cudaMemcpyFromSymbol(out3, g_order_counts, sizeof(unsigned long long) * 3));
  const unsigned long long zero[3] = {0, 0, 0};
  HG_CUDA(cudaMemcpyToSymbol(g_order_counts, zero, sizeof(zero)));
  return HG_OK;
}
