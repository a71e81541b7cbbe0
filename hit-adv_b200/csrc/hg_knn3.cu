// hg_knn3.cu -- streaming k-nearest-neighbour selection for 3-D points (KNNDist, DGCNN layer 1, knn_points).
//
// Per (query, candidate) pair the reference's distance is the same 5 FMA-pipe operations as in the Chamfer kernel
// (FMUL, 2 FFMA, 2 FADD, issued packed as FMUL2/FFMA2/FADD2 over two CANDIDATES at a time; the self-kNN path filters
// with a 4-operation folded form, see filter_addend); what differs is the selection.
// A sorted-insertion test per pair would make every warp take the slow path on almost every candidate
// (32 lanes x QT queries, each inserting ~k ln(N/k) times), and even a compare per pair costs issue slots the
// FMA pipe cannot hide on this part (FMNMX + FSETP + SEL ~ 5 slots next to 10.5 for the arithmetic, see
// profiles/r01_ubench_instruction_costs.txt).  So selection is split in two:
//   * main loop (uniform, no divergence): the threshold is folded into the last addition (filter_addend), so
//     the SIGN BIT of the result says "below this query's threshold"; the sign bits of a group of GP candidate
//     pairs are OR-ed (one LOP3 per pair) and shifted into a per-query 32-bit mask (one SHF per group);
//   * drain (divergent, rare): after each window every lane walks its flagged groups, re-evaluates the group to
//     find which candidates are below the threshold, evaluates those exactly (knn_dist_exact) and inserts them
//     into its sorted list, then refreshes the thresholds.
// With cold thresholds (no seed) the first windows are short (1, 1, 2, 4, 8 ... groups) so that the thresholds
// tighten geometrically and the number of stale hits stays ~k per doubling.
// Lists live in registers (statically indexed; KM = 6 / 20 / 32 entries, the first k are written out).
//
// Order of visits per query is ascending candidate index (sub-tiles ascending, bits ascending), insertion is
// strict '<' => equal values keep the lowest index first: the canonical tie order of the oracle.
#include "hg_common.cuh"

#include <type_traits>

namespace {

constexpr int kThreads = 128;

#define HG_KNN_FORM_EXPANDED 0  // dist = (xx_j + (-2 zz)) + xx_i   (KNNDist / DGCNN)
#define HG_KNN_FORM_DIRECT 1    // dist = fma(dz,dz, fma(dy,dy, dx*dx))   (pytorch3d knn_points)
// internal third form (see filter_addend): EXPANDED values and indices, 4-operation folded filter
#define HG_KNN_FORM_EXPANDED_FOLD4 2
__host__ __device__ constexpr bool knn_form_expanded(int form) { return form != HG_KNN_FORM_DIRECT; }

// exact scalar distance, identical operation sequence to the packed main loop
template <int FORM>
__device__ __forceinline__ float knn_dist_exact(float a0, float a1, float a2, float a3, float c0, float c1, float c2,
                                                float cw) {
  if (knn_form_expanded(FORM)) {  // a = (-2q0,-2q1,-2q2, xx_i), cw = xx_j
    const float nzz = __fmaf_rn(a2, c2, __fmaf_rn(a1, c1, __fmul_rn(a0, c0)));  // == -2*zz exactly
    return __fadd_rn(__fadd_rn(cw, nzz), a3);
  } else {  // a = (q0,q1,q2,-), c = NEGATED candidate: d = fma(dz,dz, fma(dy,dy, dx*dx)), dx = q0 + (-c0)
    const float dx = __fadd_rn(a0, c0), dy = __fadd_rn(a1, c1), dz = __fadd_rn(a2, c2);
    return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
  }
}

// exact distance for the threshold seeds: a NaN distance (a non-finite coordinate) never enters a list, so it counts as
// +inf here.  Left as NaN it would break the min/max insertion networks below (fminf / fmaxf drop it and the level
// duplicates its entry, leaving a bound under the true k-th value) and the max of the temporal seeds (a bound resting
// on k1 - 1 real candidates).
__device__ __forceinline__ float knn_seed_dist(float a0, float a1, float a2, float a3, float c0, float c1, float c2,
                                               float cw) {
  const float d = knn_dist_exact<HG_KNN_FORM_EXPANDED>(a0, a1, a2, a3, c0, c1, c2, cw);
  return d == d ? d : CUDART_INF_F;
}

// The main loop never needs the distance itself, only whether it is below the query's threshold -- and that test
// can be folded into the last addition.  EXPANDED: d = fl(s + a3) with s = fl(cw + nzz); with the addend
// af = rd(a3 - thr) the sign bit of fl(s + af) is set iff s < ru(thr - a3) (a sum of two floats never rounds to
// zero, and an exactly-zero sum is +0), and s >= ru(thr - a3) >= thr - a3 implies fl(s + a3) >= thr by
// monotonicity of rounding: no candidate below the threshold is missed; the few extra flags (within one ulp of
// the threshold) are rejected by the exact re-evaluation in the drain.  DIRECT: fl(d - thr) < 0 iff d < thr.
// A +inf threshold gives af = -inf: every finite candidate is flagged; padding (s = +inf) gives NaN, sign clear.
// Internal third form: EXPANDED arithmetic for everything that decides a value or an index, but a FOUR-operation
// filter: e = fma(a0,c0, fma(a1,c1, fma(a2,c2, cw + af))), af = rd(a3 - T), T = thr + slack.  It is not the reference's
// operation order, so it may differ from fl(s + a3) - thr by rounding: with u = 2^-24 and S = (|q| + max|c|)^2,
//   |fl-chain(reference) - R| <= 8 u S   and   |e - (R - T)| <= 5 u (S + T)      (R = the exact real distance),
// hence d < thr  =>  e < -slack + 8uS + 5u(S + T) < 0 once slack >= 24 u (S + thr) = 1.5e-6 (S + thr): nothing below
// the threshold is missed; what the slack lets through extra (a relative 1e-6 band) dies in the exact drain.
// Needs an upper bound on max|c|^2 per cloud (sbound); used on the seeded self-kNN path, where the grid pre-pass
// has the bounding box anyway.

template <int FORM>
__device__ __forceinline__ float filter_addend(float a3, float thr, float S) {
  if (FORM == HG_KNN_FORM_EXPANDED) return __fsub_rd(a3, thr);
  if (FORM == HG_KNN_FORM_EXPANDED_FOLD4) return __fsub_rd(a3, __fadd_ru(thr, 1.5e-6f * (S + thr)));
  return -thr;
}

// packed filter value of one candidate pair (A = (c0_j, c0_j1, c1_j, c1_j1), B = (c2_j, c2_j1, w_j, w_j1)).
// EXPANDED / DIRECT: same operation sequence as knn_dist_exact except that the last addend carries the threshold.
template <int FORM>
__device__ __forceinline__ float2 filter_value(float a0, float a1, float a2, float af, float4 cA, float4 cB) {
  if (FORM == HG_KNN_FORM_EXPANDED) {
    float2 tt = __fmul2_rn(make_float2(a0, a0), make_float2(cA.x, cA.y));
    tt = __ffma2_rn(make_float2(a1, a1), make_float2(cA.z, cA.w), tt);
    tt = __ffma2_rn(make_float2(a2, a2), make_float2(cB.x, cB.y), tt);
    const float2 s = __fadd2_rn(make_float2(cB.z, cB.w), tt);
    return __fadd2_rn(s, make_float2(af, af));
  } else if (FORM == HG_KNN_FORM_EXPANDED_FOLD4) {
    float2 tt = __fadd2_rn(make_float2(cB.z, cB.w), make_float2(af, af));
    tt = __ffma2_rn(make_float2(a2, a2), make_float2(cB.x, cB.y), tt);
    tt = __ffma2_rn(make_float2(a1, a1), make_float2(cA.z, cA.w), tt);
    return __ffma2_rn(make_float2(a0, a0), make_float2(cA.x, cA.y), tt);
  } else {
    const float2 dx = __fadd2_rn(make_float2(a0, a0), make_float2(cA.x, cA.y));
    const float2 dy = __fadd2_rn(make_float2(a1, a1), make_float2(cA.z, cA.w));
    const float2 dz = __fadd2_rn(make_float2(a2, a2), make_float2(cB.x, cB.y));
    const float2 d = __ffma2_rn(dz, dz, __ffma2_rn(dy, dy, __fmul2_rn(dx, dx)));
    return __fadd2_rn(d, make_float2(af, af));
  }
}

// Sorted list held in registers (static indexing only).  Candidates reach a query in ascending index order; a
// candidate enters only if strictly smaller than the current last element and bubbles up while strictly
// smaller than its predecessor => lowest index first on ties.
template <int KM>
struct TopK {
  float v[KM];
  int id[KM];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int t = 0; t < KM; ++t) {
      v[t] = CUDART_INF_F;
      id[t] = 0;
    }
  }
  __device__ __forceinline__ void push(float d, int j) {
    if (d < v[KM - 1]) {
      v[KM - 1] = d;
      id[KM - 1] = j;
#pragma unroll
      for (int t = KM - 1; t > 0; --t) {
        if (v[t] < v[t - 1]) {
          const float tv = v[t];
          v[t] = v[t - 1];
          v[t - 1] = tv;
          const int ti = id[t];
          id[t] = id[t - 1];
          id[t - 1] = ti;
        }
      }
    }
  }
};

// Drain of flagged group grp of the staged pairs (candidates base + 2*GP*grp ...): the group is re-evaluated with the
// same packed filter arithmetic to find WHICH of its 2*GP candidates are below the threshold, and only those are
// evaluated exactly and inserted.  The insertion code (the expensive part) is thus reached once per group by all lanes
// together, not once per candidate slot.
template <int FORM, int KM, int GP>
__device__ __forceinline__ void knn_drain_group(float a0, float a1, float a2, float a3, float af, TopK<KM> &top,
                                                const float4 *cand, int grp, int base) {
  const float4 *cp = cand + 2 * GP * grp;
  unsigned sub = 0u;  // after 2*GP shifts, bit 2*GP-1-c belongs to candidate c of the group
#pragma unroll
  for (int u = 0; u < GP; ++u) {
    const float4 cA = cp[2 * u], cB = cp[2 * u + 1];
    const float2 e = filter_value<FORM>(a0, a1, a2, af, cA, cB);
    sub = __funnelshift_l(__float_as_uint(e.x), sub, 1);
    sub = __funnelshift_l(__float_as_uint(e.y), sub, 1);
  }
  while (sub) {
    const int sp = 31 - __clz(sub);
    sub &= ~(1u << sp);
    const int c = 2 * GP - 1 - sp;
    const float4 cA = cp[2 * (c >> 1)], cB = cp[2 * (c >> 1) + 1];
    const bool hi = c & 1;
    top.push(knn_dist_exact<FORM>(a0, a1, a2, a3, hi ? cA.y : cA.x, hi ? cA.w : cA.z, hi ? cB.y : cB.x, hi ? cB.w : cB.z),
             base + 2 * GP * grp + c);
  }
}

// the first k1 entries of query i's list (nothing past Nq); idx_state, when given, gets a second copy of the indices
template <int KM, typename IdxT>
__device__ __forceinline__ void knn_write_list(const TopK<KM> &top, int b, int i, int Nq, int k1, float *vals, IdxT *idx,
                                               int *idx_state) {
  if (i < Nq) {
#pragma unroll
    for (int s = 0; s < KM; ++s) {
      if (s < k1) {
        if (vals) vals[((size_t)b * Nq + i) * k1 + s] = top.v[s];
        idx[((size_t)b * Nq + i) * k1 + s] = (IdxT)top.id[s];
        if (idx_state) idx_state[((size_t)b * Nq + i) * k1 + s] = top.id[s];
      }
    }
  }
}

// KM >= k1 list entries are kept; the first k1 are written out.
// GP = candidate pairs per hit bit; a tile is 32 groups (one 32-bit mask per query) = 64*GP candidates.
template <int FORM, int QT, int KM, int GP, typename IdxT>
__global__ void __launch_bounds__(kThreads) knn3_kernel(const float *__restrict__ queries,
                                                        const float *__restrict__ refs, int Nq, int Nr, int k1,
                                                        float *__restrict__ vals, IdxT *__restrict__ idx,
                                                        const float *__restrict__ thr0 /*[B,Nq] or null*/,
                                                        const float *__restrict__ sbound /*FOLD4: [B] stride 8,
                                                        upper bound on max |candidate|^2*/,
                                                        int *__restrict__ idx_state /*second copy of idx or null*/,
                                                        const float4 *__restrict__ only /*null, or per-cloud info of
                                                        a pruned-path ordering: flagged clouds only*/) {
  if (only != nullptr && only[blockIdx.y].y == 0.f) return;
  constexpr int kTilePairs = 32 * GP;
  constexpr int kTileC = 2 * kTilePairs;
  __shared__ float4 cand[2 * kTilePairs];  // two float4 per candidate pair
  const int b = blockIdx.y, tid = threadIdx.x;
  const float *q = queries + (size_t)b * Nq * 3;
  const float *r = refs + (size_t)b * Nr * 3;

  float a0[QT], a1[QT], a2[QT], a3[QT], af[QT], seed[QT], S[QT];
  const float cmax = (FORM == HG_KNN_FORM_EXPANDED_FOLD4) ? sqrtf(sbound[(size_t)b * 8]) : 0.f;
  unsigned mask[QT];
  TopK<KM> top[QT];
#pragma unroll
  for (int t = 0; t < QT; ++t) {
    const int i = (blockIdx.x * QT + t) * kThreads + tid;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
    if (i < Nq) {
      q0 = __ldg(q + (size_t)i * 3);
      q1 = __ldg(q + (size_t)i * 3 + 1);
      q2 = __ldg(q + (size_t)i * 3 + 2);
    }
    if (knn_form_expanded(FORM)) {
      a0[t] = -2.0f * q0;
      a1[t] = -2.0f * q1;
      a2[t] = -2.0f * q2;
      a3[t] = hg_sumsq3_seq(q0, q1, q2);
    } else {
      a0[t] = q0;
      a1[t] = q1;
      a2[t] = q2;
      a3[t] = 0.f;
    }
    // optional upper bound on this query's KM-th distance (knn_seed_kernel): the filter starts tight instead of
    // at +inf, so only ~KM candidates ever reach the drain instead of ~KM ln(N/KM)
    seed[t] = (thr0 != nullptr && i < Nq) ? thr0[(size_t)b * Nq + i] : CUDART_INF_F;
    S[t] = (sqrtf(a3[t]) + cmax) * (sqrtf(a3[t]) + cmax) * 1.0001f;
    af[t] = filter_addend<FORM>(a3[t], seed[t], S[t]);
    mask[t] = 0u;
    top[t].init();
  }

  for (int base = 0; base < Nr; base += kTileC) {
    __syncthreads();
    // stage the tile as candidate PAIRS: A = (c0_j, c0_j1, c1_j, c1_j1), B = (c2_j, c2_j1, w_j, w_j1)
    for (int p = tid; p < kTilePairs; p += kThreads) {
      float c[2][4];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = base + 2 * p + h;
        c[h][0] = c[h][1] = c[h][2] = 0.f;
        c[h][3] = CUDART_INF_F;  // padding can never beat a threshold (EXPANDED: inf; DIRECT: handled below)
        if (j < Nr) {
          const float x = __ldg(r + (size_t)j * 3), y = __ldg(r + (size_t)j * 3 + 1), z = __ldg(r + (size_t)j * 3 + 2);
          if (knn_form_expanded(FORM)) {
            c[h][0] = x; c[h][1] = y; c[h][2] = z;
            c[h][3] = hg_sumsq3_seq(x, y, z);
          } else {
            c[h][0] = -x; c[h][1] = -y; c[h][2] = -z;
            c[h][3] = 0.f;
          }
        } else if (!knn_form_expanded(FORM)) {
          c[h][0] = CUDART_INF_F;  // dx = q + inf = inf -> d = inf
        }
      }
      cand[2 * p] = make_float4(c[0][0], c[1][0], c[0][1], c[1][1]);
      cand[2 * p + 1] = make_float4(c[0][2], c[1][2], c[0][3], c[1][3]);
    }
    __syncthreads();
    const int ngroups = ((min(kTileC, Nr - base) + 1) / 2 + GP - 1) / GP;

    // Windows between two drains, in groups.  First tile: 1,1,2,4,8,8,8 groups so that cold thresholds tighten
    // geometrically.  Later tiles: the whole tile in one window -- hits are rare per lane but frequent per warp
    // there, and a longer window lets several lanes insert in the same (divergent) drain iteration.
    int g0 = 0;
    int step = (base == 0) ? 1 : 32;
    while (g0 < ngroups) {
      const int cnt = min(step, ngroups - g0);
      // ---- main loop: packed filter values, sign bits OR-ed per group and shifted into the query's mask ------
      // (after cnt shifts, bit cnt-1-g belongs to group g0+g)
#pragma unroll (KM <= 6 ? 2 : 1)
      for (int g = 0; g < cnt; ++g) {
        const float4 *cp = cand + 2 * GP * (g0 + g);
        float4 cA[GP], cB[GP];
#pragma unroll
        for (int u = 0; u < GP; ++u) {
          cA[u] = cp[2 * u];
          cB[u] = cp[2 * u + 1];
        }
#pragma unroll
        for (int t = 0; t < QT; ++t) {
          unsigned o = 0u;
#pragma unroll
          for (int u = 0; u < GP; ++u) {
            const float2 e = filter_value<FORM>(a0[t], a1[t], a2[t], af[t], cA[u], cB[u]);
            o |= __float_as_uint(e.x) | __float_as_uint(e.y);
          }
          mask[t] = __funnelshift_l(o, mask[t], 1);
        }
      }
      // ---- drain (divergent, rare).  Each lane walks its flagged groups in ascending order; a group is
      // re-evaluated with the same packed filter arithmetic to find WHICH of its 2*GP candidates are below the
      // threshold, and only those are evaluated exactly and inserted.  The insertion code (the expensive part)
      // is thus reached once per group iteration by all lanes together, not once per candidate slot.
#pragma unroll
      for (int t = 0; t < QT; ++t) {
        unsigned m = mask[t];
        while (m) {
          const int pos = 31 - __clz(m);
          m &= ~(1u << pos);
          const int grp = g0 + cnt - 1 - pos;
          knn_drain_group<FORM, KM, GP>(a0[t], a1[t], a2[t], a3[t], af[t], top[t], cand, grp, base);
        }
        mask[t] = 0u;
        af[t] = filter_addend<FORM>(a3[t], fminf(seed[t], top[t].v[KM - 1]), S[t]);
      }
      g0 += cnt;
      if (base == 0 && step < 8 && g0 >= 2 * step) step *= 2;  // 1,1,2,4,8,8,8
    }
  }

#pragma unroll
  for (int t = 0; t < QT; ++t)
    knn_write_list(top[t], b, (blockIdx.x * QT + t) * kThreads + tid, Nq, k1, vals, idx, idx_state);
}

// ---- small clouds (< 2k points): whole candidate set resident in shared memory, drain deferred -----------------
// At 1024 points the streaming kernel above spends more time in its per-tile drains than in its main loop: with 8
// tiles, every tile ends in a divergent drain that lasts as long as the unluckiest lane's hits, and the cold
// thresholds of the first tile flag most candidates.  Here
//   * every query starts from an exact upper bound on its k-th distance (knn_seed_small_kernel: a uniform grid built
//     in shared memory by one CTA per cloud), so the filter is tight from the first candidate;
//   * the whole cloud is staged once (16 B per candidate), the main loop runs over ALL candidate pairs without a
//     barrier or a drain, storing one mask word per 32 groups in shared memory;
//   * ONE drain at the end walks the flagged groups of all words in a single loop: its length is the largest number of
//     flagged groups any lane has in total, not the sum over tiles of the per-tile maxima.
// A word in which some lane flags more than kDrainNow groups (a loose or infinite seed) triggers an immediate drain,
// which tightens that lane's threshold, so correctness and progress never depend on the quality of the seeds.
constexpr int kDrainNow = 12;

template <int QT, int KM, int GP>
__global__ void __launch_bounds__(kThreads) knn3_small_kernel(const float *__restrict__ pc, int N, int k1, int W,
                                                              float *__restrict__ vals, int *__restrict__ idx,
                                                              const float *__restrict__ thr0 /*[B,N]*/,
                                                              const float *__restrict__ sbound /*[B] stride 8*/,
                                                              int *__restrict__ idx_state /*second copy or null*/) {
  constexpr int FORM = HG_KNN_FORM_EXPANDED_FOLD4;
  extern __shared__ float4 smem4[];
  const int npairs = W * 32 * GP;               // padded to whole mask words
  float4 *cand = smem4;                         // two float4 per candidate pair
  unsigned *smask = reinterpret_cast<unsigned *>(cand + 2 * (size_t)npairs);  // [QT][W][kThreads]
  const int b = blockIdx.y, tid = threadIdx.x;
  const float *p = pc + (size_t)b * N * 3;

  for (int pr = tid; pr < npairs; pr += kThreads) {
    float c[2][4];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * pr + h;
      c[h][0] = c[h][1] = c[h][2] = 0.f;
      c[h][3] = CUDART_INF_F;
      if (j < N) {
        const float x = __ldg(p + (size_t)j * 3), y = __ldg(p + (size_t)j * 3 + 1), z = __ldg(p + (size_t)j * 3 + 2);
        c[h][0] = x; c[h][1] = y; c[h][2] = z;
        c[h][3] = hg_sumsq3_seq(x, y, z);
      }
    }
    cand[2 * pr] = make_float4(c[0][0], c[1][0], c[0][1], c[1][1]);
    cand[2 * pr + 1] = make_float4(c[0][2], c[1][2], c[0][3], c[1][3]);
  }

  float a0[QT], a1[QT], a2[QT], a3[QT], af[QT], seed[QT], S[QT];
  unsigned nz[QT];
  TopK<KM> top[QT];
  const float cmax = sqrtf(sbound[(size_t)b * 8]);
#pragma unroll
  for (int t = 0; t < QT; ++t) {
    const int i = (blockIdx.x * QT + t) * kThreads + tid;
    float q0 = 0.f, q1 = 0.f, q2 = 0.f;
    if (i < N) {
      q0 = __ldg(p + (size_t)i * 3);
      q1 = __ldg(p + (size_t)i * 3 + 1);
      q2 = __ldg(p + (size_t)i * 3 + 2);
    }
    a0[t] = -2.0f * q0;
    a1[t] = -2.0f * q1;
    a2[t] = -2.0f * q2;
    a3[t] = hg_sumsq3_seq(q0, q1, q2);
    seed[t] = (i < N) ? thr0[(size_t)b * N + i] : -CUDART_INF_F;  // lanes past the cloud never flag anything
    S[t] = (sqrtf(a3[t]) + cmax) * (sqrtf(a3[t]) + cmax) * 1.0001f;
    af[t] = filter_addend<FORM>(a3[t], seed[t], S[t]);
    nz[t] = 0u;
    top[t].init();
  }
  __syncthreads();

  // flagged groups of the pending words of query t, ascending; thresholds refreshed after every group.  The group drain
  // (and the staging, query set-up and filter above) repeat knn3_kernel's: the shared helpers compile to different
  // machine code for this kernel, knn_drain_group included.
  auto drain = [&](int t) {
    unsigned pend = nz[t], m = 0u;
    int w = 0;
    while (true) {
      if (m == 0u) {
        if (pend == 0u) break;
        w = __ffs(pend) - 1;
        pend &= pend - 1u;
        m = smask[((size_t)t * W + w) * kThreads + tid];  // non-zero by construction
      }
      const int pos = 31 - __clz(m);
      m &= ~(1u << pos);
      const int grp = w * 32 + (31 - pos);
      const float4 *cp = cand + 2 * GP * grp;
      unsigned sub = 0u;  // after 2*GP shifts, bit 2*GP-1-c belongs to candidate c of the group
#pragma unroll
      for (int u = 0; u < GP; ++u) {
        const float4 cA = cp[2 * u], cB = cp[2 * u + 1];
        const float2 e = filter_value<FORM>(a0[t], a1[t], a2[t], af[t], cA, cB);
        sub = __funnelshift_l(__float_as_uint(e.x), sub, 1);
        sub = __funnelshift_l(__float_as_uint(e.y), sub, 1);
      }
      while (sub) {
        const int sp = 31 - __clz(sub);
        sub &= ~(1u << sp);
        const int c = 2 * GP - 1 - sp;
        const float4 cA = cp[2 * (c >> 1)], cB = cp[2 * (c >> 1) + 1];
        const bool hi = c & 1;
        top[t].push(knn_dist_exact<FORM>(a0[t], a1[t], a2[t], a3[t], hi ? cA.y : cA.x, hi ? cA.w : cA.z,
                                         hi ? cB.y : cB.x, hi ? cB.w : cB.z),
                    2 * GP * grp + c);
      }
      af[t] = filter_addend<FORM>(a3[t], fminf(seed[t], top[t].v[KM - 1]), S[t]);
    }
    nz[t] = 0u;
  };

  for (int w = 0; w < W; ++w) {
    unsigned mk[QT];
#pragma unroll
    for (int t = 0; t < QT; ++t) mk[t] = 0u;
    const float4 *wp = cand + (size_t)2 * GP * 32 * w;
#pragma unroll (KM <= 6 ? 2 : 1)
    for (int g = 0; g < 32; ++g) {
      const float4 *cp = wp + 2 * GP * g;
      float4 cA[GP], cB[GP];
#pragma unroll
      for (int u = 0; u < GP; ++u) {
        cA[u] = cp[2 * u];
        cB[u] = cp[2 * u + 1];
      }
#pragma unroll
      for (int t = 0; t < QT; ++t) {
        unsigned o = 0u;
#pragma unroll
        for (int u = 0; u < GP; ++u) {
          const float2 e = filter_value<FORM>(a0[t], a1[t], a2[t], af[t], cA[u], cB[u]);
          o |= __float_as_uint(e.x) | __float_as_uint(e.y);
        }
        mk[t] = __funnelshift_l(o, mk[t], 1);  // after 32 shifts, bit 31-g belongs to group g of this word
      }
    }
    bool crowded = false;
#pragma unroll
    for (int t = 0; t < QT; ++t) {
      smask[((size_t)t * W + w) * kThreads + tid] = mk[t];
      if (mk[t]) nz[t] |= 1u << w;
      crowded |= __popc(mk[t]) > kDrainNow;
    }
    if (__any_sync(0xffffffffu, crowded)) {
#pragma unroll
      for (int t = 0; t < QT; ++t) drain(t);
    }
  }
#pragma unroll
  for (int t = 0; t < QT; ++t) drain(t);

#pragma unroll
  for (int t = 0; t < QT; ++t)
    knn_write_list(top[t], b, (blockIdx.x * QT + t) * kThreads + tid, N, k1, vals, idx, idx_state);
}

// Seeds for the small-cloud kernel.  One CTA per cloud sorts the cloud along a Z-order (Morton) curve in shared memory
// -- bounding box, 12-bit Morton cell of every point (16 cells per axis), counting sort by cell -- and every query takes
// the k1-th smallest distance over the `win` points around its own position in that order (itself included),
// evaluated with the main kernel's exact arithmetic.  Those are real candidates, hence an exact upper bound on the
// query's k1-th distance (nudged one ulp so that the strict '<' of the filter keeps ties); a window in Z-order adapts
// to the local density, where a fixed neighbourhood of grid cells is empty in the tails of a cloud and crowded at its
// centre.  Any bound would be CORRECT -- the main kernel drains early when a bound is loose -- a good one keeps it fast.
constexpr int kMortonBits = 4, kMortonCells = 1 << (3 * kMortonBits);

// Upper bound on max |p|^2 over a bounding box whose lo x, y, z, hi x, y, z lie `stride` floats apart: its farthest
// corner, widened for rounding (the folded filter's slack needs it)
__device__ __forceinline__ float knn_box_sbound(const float *box, int stride) {
  float sb = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) sb += fmaxf(box[c * stride] * box[c * stride], box[(3 + c) * stride] * box[(3 + c) * stride]);
  return sb * 1.0001f;
}

// sbound[b * 8] = the largest m of a 256-thread CTA (each thread's bound on max |p|^2 over its points), widened for rounding
__device__ __forceinline__ void knn_block_sbound(float m, int tid, float *sbound, int b) {
  __shared__ float red[8];
  m = hg_warp_max_f32(m);
  if ((tid & 31) == 0) red[tid >> 5] = m;
  __syncthreads();
  if (tid == 0) {
    for (int w = 1; w < 8; ++w) m = fmaxf(m, red[w]);
    sbound[(size_t)b * 8] = m * 1.0001f;
  }
}

__device__ __forceinline__ int morton3_4bit(int x, int y, int z) {
  auto spread = [](int v) { return (v & 1) | ((v & 2) << 2) | ((v & 4) << 4) | ((v & 8) << 6); };
  return spread(x) | (spread(y) << 1) | (spread(z) << 2);
}

template <int KM>
__global__ void __launch_bounds__(256) knn_seed_small_kernel(const float *__restrict__ pc, int N, int k1, int win,
                                                             float *__restrict__ thr0, float *__restrict__ sbound) {
  extern __shared__ float4 spts[];                   // [N] (x, y, z, xx) in Z-order
  int *sidx = reinterpret_cast<int *>(spts + N);     // [N] original index of the point at each sorted position
  int *scr = sidx + N;                               // [N] cell | rank-within-cell << 12
  __shared__ int soff[kMortonCells + 1];
  __shared__ float sred[6][8];
  __shared__ float sbox[6];
  __shared__ int swsum[8];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float *p = pc + (size_t)b * N * 3;

  float lo[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, hi[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  for (int i = tid; i < N; i += 256)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = __ldg(p + (size_t)i * 3 + c);
      lo[c] = fminf(lo[c], v);
      hi[c] = fmaxf(hi[c], v);
    }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    lo[c] = hg_warp_min_f32(lo[c]);
    hi[c] = hg_warp_max_f32(hi[c]);
  }
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      sred[c][warp] = lo[c];
      sred[3 + c][warp] = hi[c];
    }
  for (int c = tid; c <= kMortonCells; c += 256) soff[c] = 0;
  __syncthreads();
  if (tid < 6) {
    float v = sred[tid][0];
    for (int w = 1; w < 8; ++w) v = tid < 3 ? fminf(v, sred[tid][w]) : fmaxf(v, sred[tid][w]);
    sbox[tid] = v;
  }
  __syncthreads();
  float mn[3], inv[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    mn[c] = sbox[c];
    const float ext = sbox[3 + c] - mn[c];
    inv[c] = (ext > 0.f && ext < CUDART_INF_F) ? (float)(1 << kMortonBits) / ext : 0.f;
  }
  if (tid == 0) sbound[(size_t)b * 8] = knn_box_sbound(sbox, 1);
  for (int i = tid; i < N; i += 256) {
    int cc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float f = (__ldg(p + (size_t)i * 3 + c) - mn[c]) * inv[c];
      cc[c] = (f == f) ? min(max((int)f, 0), (1 << kMortonBits) - 1) : 0;
    }
    const int cell = morton3_4bit(cc[0], cc[1], cc[2]);
    const int rank = atomicAdd(&soff[cell], 1);  // order within a cell is irrelevant to a k-th smallest VALUE
    scr[i] = cell | (rank << 12);
  }
  __syncthreads();
  {  // exclusive scan of the 4096 cell counts: 16 consecutive cells per thread, then a block scan of the thread sums
    constexpr int per = kMortonCells / 256;
    int cnt[per], sum = 0;
#pragma unroll
    for (int c = 0; c < per; ++c) {
      cnt[c] = soff[tid * per + c];
      sum += cnt[c];
    }
    int incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int o = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += o;
    }
    if (lane == 31) swsum[warp] = incl;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; ++w) base += swsum[w];
    int run = base + incl - sum;
#pragma unroll
    for (int c = 0; c < per; ++c) {
      soff[tid * per + c] = run;
      run += cnt[c];
    }
  }
  __syncthreads();
  for (int i = tid; i < N; i += 256) {
    const float x = __ldg(p + (size_t)i * 3), y = __ldg(p + (size_t)i * 3 + 1), z = __ldg(p + (size_t)i * 3 + 2);
    const int v = scr[i];
    const int pos = soff[v & (kMortonCells - 1)] + (v >> 12);
    spts[pos] = make_float4(x, y, z, hg_sumsq3_seq(x, y, z));
    sidx[pos] = i;
  }
  __syncthreads();

  // queries in Z-order: the windows of the 32 lanes of a warp overlap (consecutive shared-memory addresses)
  for (int s = tid; s < N; s += 256) {
    const float4 q = spts[s];
    const float a0 = -2.0f * q.x, a1 = -2.0f * q.y, a2 = -2.0f * q.z, a3 = q.w;
    float v[KM];
#pragma unroll
    for (int t = 0; t < KM; ++t) v[t] = CUDART_INF_F;
    const int t0 = max(0, min(s - win / 2, N - win)), t1 = min(N, t0 + win);
    for (int t = t0; t < t1; ++t) {
      const float4 r = spts[t];
      hg_sorted_min_insert(v, knn_seed_dist(a0, a1, a2, a3, r.x, r.y, r.z, r.w));
    }
    float bound = -CUDART_INF_F;  // v[k1-1] = the largest of the first k1 entries (v is ascending); written as a max
#pragma unroll                    // so that the list stays in registers (a runtime index would move it to local memory)
    for (int t = 0; t < KM; ++t)
      if (t < k1) bound = fmaxf(bound, v[t]);
    thr0[(size_t)b * N + sidx[s]] = hg_nudge_up(bound);
  }
}

// Test-only override of the instantiation launch_form / launch_qt would pick from the problem size (0 = automatic):
// lets small seeded inputs reach every (QT, GP) variant, including the ones only large batches select.
static int g_force_qt = 0, g_force_gp = 0;

// k1 -> the list length KM that serves it: f(std::integral_constant<int, KM>{}) with KM = 6, 20, 32 and, for kernels
// instantiated with lists of 64, 64
template <int kMaxKM, typename F>
auto with_km(int k1, F &&f) {
  if (k1 <= 6) return f(std::integral_constant<int, 6>{});
  if (k1 <= 20) return f(std::integral_constant<int, 20>{});
  if constexpr (kMaxKM > 32) {
    if (k1 > 32) return f(std::integral_constant<int, 64>{});
  }
  return f(std::integral_constant<int, 32>{});
}

// One dispatch over the instantiated (KM, QT) set of both kNN kernels: up to 4 queries per lane with 6-entry lists, 2
// with 20, 1 beyond.  A QT outside it (forced through hg_knn_force_shape) is an error.
template <int kMaxKM, typename F>
int with_km_qt(int k1, int qt, F &&f) {
  return with_km<kMaxKM>(k1, [&](auto km) -> int {
    constexpr int KM = decltype(km)::value;
    if (qt == 1) return f(km, std::integral_constant<int, 1>{});
    if constexpr (KM <= 20) {
      if (qt == 2) return f(km, std::integral_constant<int, 2>{});
    }
    if constexpr (KM <= 6) {
      if (qt == 4) return f(km, std::integral_constant<int, 4>{});
    }
    hg_set_error("knn: forced QT=%d has no instantiation for k=%d", qt, k1);
    return HG_E_UNSUPPORTED;
  });
}

template <int FORM, int QT, int KM, typename IdxT>
int launch_qt(const float *q, const float *r, int B, int Nq, int Nr, int k1, float *vals, IdxT *idx,
              const float *thr0, const float *sbound, cudaStream_t stream, int *idx_state = nullptr,
              const float4 *only = nullptr) {
  dim3 grid((Nq + QT * kThreads - 1) / (QT * kThreads), B);
  const bool prof = hg_prof_begin(HG_PROF_KNN, stream);
  // 8 candidates per hit bit (512-candidate tiles) for long candidate lists, 4 (256) for short ones, where the
  // cheaper group re-evaluation in the drain outweighs the extra mask updates (measured cross-over ~2-4k)
  if (g_force_gp ? g_force_gp == 2 : Nr < 2048)
    knn3_kernel<FORM, QT, KM, 2, IdxT><<<grid, kThreads, 0, stream>>>(q, r, Nq, Nr, k1, vals, idx, thr0, sbound, idx_state, only);
  else
    knn3_kernel<FORM, QT, KM, 4, IdxT><<<grid, kThreads, 0, stream>>>(q, r, Nq, Nr, k1, vals, idx, thr0, sbound, idx_state, only);
  hg_prof_end(HG_PROF_KNN, stream, prof);
  HG_CHECK_LAUNCH("knn3_kernel");
  return HG_OK;
}

template <int FORM, typename IdxT>
int launch_form(const float *q, const float *r, int B, int Nq, int Nr, int k1, float *vals, IdxT *idx,
                const float *thr0, const float *sbound, cudaStream_t stream, int *idx_state = nullptr,
                const float4 *only = nullptr) {
  if (k1 < 1 || k1 > 64) {
    hg_set_error("knn: k=%d outside [1,64]", k1);
    return HG_E_UNSUPPORTED;
  }
  // Queries per lane (QT): more queries amortise the candidate loads (LDS per pair halves with every doubling), which
  // pays on long candidate lists; on short ones (< 2k candidates) the cold-start drains dominate and run one query
  // after the other, so fewer queries per lane win (measured, k+1 = 6: 16384 points 5.96 / 6.33 / 8.72 ms for QT = 4 /
  // 2 / 1; 1024 points 2.46 / 2.14 / 2.28 ms).  Small batches additionally drop QT until the grid fills the machine.
  int qt = g_force_qt;
  if (!qt) {
    const long long want = 2LL * hg_sm_count();
    auto ctas = [&](int qt) { return (long long)B * ((Nq + qt * kThreads - 1) / (qt * kThreads)); };
    const bool short_list = Nr < 2048;
    qt = 1;
    if (k1 <= 6) {
      // (four queries per lane need twice the CTAs to pay: 32 x 8192: 654 us with two against 695, 16 x 16384: 1080 / 1128;
      // 64 x 8192 and up: four win -- tools/debug/knn_small_shapes.py big)
      if (!short_list && Nq >= 3 * kThreads && ctas(4) >= 2 * want)
        qt = 4;
      else if (Nq > kThreads && ctas(2) >= want)
        qt = 2;
    } else if (k1 <= 20 && !short_list && Nq > kThreads && ctas(2) >= want) {
      qt = 2;
    }
  }
  // 33..64 neighbours (HiT-ADV's default curv_loss_knn = 32 asks knn_points for 33): a 64-entry register list
  return with_km_qt<64>(k1, qt, [&](auto km, auto qt_) -> int {
    return launch_qt<FORM, decltype(qt_)::value, decltype(km)::value, IdxT>(q, r, B, Nq, Nr, k1, vals, idx, thr0, sbound,
                                                                            stream, idx_state, only);
  });
}

// ---- threshold seeding for self-kNN ---------------------------------------------------------------------------
// A uniform grid over the cloud's bounding box (about 3 points per cell) gives every query an exact UPPER BOUND on its
// KM-th smallest distance: the KM-th smallest over the points of its neighbouring cells (the 2x2x2 nearest ones for
// lists up to 20 entries, all 27 beyond), evaluated with the same
// expanded-form arithmetic (those points are real candidates, so the true KM-th distance cannot be larger).  The
// brute-force pass still evaluates all N^2 pairs and still decides every index itself; the seed only spares the
// ~KM ln(N/KM) insertions a cold threshold costs.  The bound is nudged up one ulp so that the strict '<' of the
// filter keeps candidates EQUAL to it.
constexpr int kMaxSeedCand = 512;

__global__ void __launch_bounds__(256) knn_cells_kernel(const float *__restrict__ pc, int N, int G,
                                                        int *__restrict__ cellid, float *__restrict__ params) {
  const int b = blockIdx.x, tid = threadIdx.x;
  const float *p = pc + (size_t)b * N * 3;
  __shared__ float red[6][256];
  float lo[3] = {CUDART_INF_F, CUDART_INF_F, CUDART_INF_F}, hi[3] = {-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F};
  for (int i = tid; i < N; i += 256)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = p[(size_t)i * 3 + c];
      lo[c] = fminf(lo[c], v);
      hi[c] = fmaxf(hi[c], v);
    }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    red[c][tid] = lo[c];
    red[3 + c][tid] = hi[c];
  }
  __syncthreads();
  for (int st = 128; st > 0; st >>= 1) {
    if (tid < st)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        red[c][tid] = fminf(red[c][tid], red[c][tid + st]);
        red[3 + c][tid] = fmaxf(red[3 + c][tid], red[3 + c][tid + st]);
      }
    __syncthreads();
  }
  float mn[3], inv[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    mn[c] = red[c][0];
    const float ext = red[3 + c][0] - mn[c];
    inv[c] = (ext > 0.f && ext < CUDART_INF_F) ? (float)G / ext : 0.f;
  }
  if (tid < 3) {
    params[b * 8 + tid] = mn[tid];
    params[b * 8 + 3 + tid] = inv[tid];
  }
  if (tid == 0) params[b * 8 + 6] = knn_box_sbound(&red[0][0], 256);
  for (int i = tid; i < N; i += 256) {
    int cc[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float f = (p[(size_t)i * 3 + c] - mn[c]) * inv[c];
      cc[c] = (f == f) ? min(max((int)f, 0), G - 1) : 0;
    }
    cellid[(size_t)b * N + i] = (cc[2] * G + cc[1]) * G + cc[0];
  }
}

// points re-ordered by cell (the CSR list is a permutation of the cloud grouped by cell): (x, y, z, xx)
__global__ void __launch_bounds__(256) knn_cell_sort_kernel(const float *__restrict__ pc, const int *__restrict__ list,
                                                            long long total, int N, float4 *__restrict__ sorted) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total;
       g += (long long)gridDim.x * blockDim.x) {
    const long long b = g / N;
    const float *p = pc + ((size_t)b * N + list[g]) * 3;
    const float x = p[0], y = p[1], z = p[2];
    sorted[g] = make_float4(x, y, z, hg_sumsq3_seq(x, y, z));
  }
}

// one thread per query, in CELL ORDER: the 32 queries of a warp sit in a handful of neighbouring cells, so their
// candidate runs (3 x-adjacent cells are contiguous in `sorted`) overlap and come from L1
template <int KM>
__global__ void __launch_bounds__(128) knn_seed_kernel(const float4 *__restrict__ sorted, int N, int G,
                                                       const float *__restrict__ params, const int *__restrict__ off,
                                                       const int *__restrict__ list, float *__restrict__ thr0,
                                                       int near8) {
  const int b = blockIdx.y, s_q = blockIdx.x * 128 + threadIdx.x;
  if (s_q >= N) return;
  const float4 *pts = sorted + (size_t)b * N;
  const int ncell = G * G * G;
  const int *o = off + (size_t)b * (ncell + 1);
  const float4 q = pts[s_q];
  const float a0 = -2.0f * q.x, a1 = -2.0f * q.y, a2 = -2.0f * q.z, a3 = q.w;
  int cc[3], lo[3], hi[3];
  const float qq[3] = {q.x, q.y, q.z};
#pragma unroll
  for (int c = 0; c < 3; ++c) {  // same expression as knn_cells_kernel -> same cell
    const float f = (qq[c] - params[b * 8 + c]) * params[b * 8 + 3 + c];
    cc[c] = (f == f) ? min(max((int)f, 0), G - 1) : 0;
    // near8: only the 2x2x2 cells nearest to the query (the neighbour on the side of the cell the query sits in)
    const int side = (f - (float)cc[c] < 0.5f) ? -1 : 1;
    lo[c] = near8 ? min(cc[c], cc[c] + side) : cc[c] - 1;
    hi[c] = near8 ? max(cc[c], cc[c] + side) : cc[c] + 1;
  }
  float v[KM];
#pragma unroll
  for (int t = 0; t < KM; ++t) v[t] = CUDART_INF_F;
  // the (up to 9) runs of x-adjacent cells: all their bounds are loaded before the first candidate (independent loads,
  // one latency instead of one per run)
  int rb[9], re[9];
  int nruns = 0;
#pragma unroll
  for (int zz = 0; zz < 3; ++zz)
#pragma unroll
    for (int yy = 0; yy < 3; ++yy) {
      const int z = lo[2] + zz, y = lo[1] + yy;
      const bool ok = z <= hi[2] && y <= hi[1] && z >= 0 && z < G && y >= 0 && y < G;
      const int x0 = max(lo[0], 0), x1 = min(hi[0], G - 1);
      const int c0 = ok ? (z * G + y) * G + x0 : 0, c1 = ok ? (z * G + y) * G + x1 : -1;
      rb[zz * 3 + yy] = ok ? o[c0] : 0;
      re[zz * 3 + yy] = ok ? o[c1 + 1] : 0;
      nruns += ok;
    }
  (void)nruns;
  int seen = 0;
#pragma unroll
  for (int rI = 0; rI < 9; ++rI) {
    int t = rb[rI];
    const int te = min(re[rI], t + (kMaxSeedCand - seen));
    seen += max(te - t, 0);
    for (; t + 1 < te; t += 2) {  // two candidates in flight; insertion without branches (values only)
      const float4 r0 = pts[t], r1 = pts[t + 1];
      const float d0 = knn_seed_dist(a0, a1, a2, a3, r0.x, r0.y, r0.z, r0.w);
      const float d1 = knn_seed_dist(a0, a1, a2, a3, r1.x, r1.y, r1.z, r1.w);
      hg_sorted_min_insert(v, d0);
      hg_sorted_min_insert(v, d1);
    }
    if (t < te) {
      const float4 r0 = pts[t];
      hg_sorted_min_insert(v, knn_seed_dist(a0, a1, a2, a3, r0.x, r0.y, r0.z, r0.w));
    }
  }
  thr0[(size_t)b * N + list[(size_t)b * N + s_q]] = hg_nudge_up(v[KM - 1]);
}

// upper bound on max |p|^2 per cloud for the folded filter when no grid pre-pass runs: sbound[b*8] (stride 8, like params+6)
__global__ void __launch_bounds__(256) knn_bound_kernel(const float *__restrict__ pc, int N, float *__restrict__ sbound) {
  const int b = blockIdx.x, tid = threadIdx.x;
  const float *p = pc + (size_t)b * N * 3;
  float m = 0.f;
  for (int i = tid; i < N; i += 256) {
    const float x = p[(size_t)i * 3], y = p[(size_t)i * 3 + 1], z = p[(size_t)i * 3 + 2];
    m = fmaxf(m, fmaf(z, z, fmaf(y, y, x * x)));
  }
  knn_block_sbound(m, tid, sbound, b);
}

// Temporal seeds (attack loops call KNNDist thousands of times on a slowly moving cloud, CW/kNN.py:77-111): the
// k1 neighbours a query had on the previous call, re-evaluated at the CURRENT coordinates with the main kernel's exact
// arithmetic, are k1 distinct real candidates, so the largest of their distances is an exact upper bound on the
// query's k1-th distance -- k1 evaluations per query instead of a spatial pre-pass, and a bound that is nearly tight.
// The saved indices are only trusted after checking them: out of range or repeated entries give an infinite bound for
// that query (it is then handled like an unseeded one), never a wrong result.  One CTA per cloud; also produces the
// bound on max |p|^2 the folded filter needs.
template <int KM>
__global__ void __launch_bounds__(256) knn_seed_prev_kernel(const float *__restrict__ pc, int N, int k1,
                                                            const int *__restrict__ prev /*[B,N,k1]*/,
                                                            float *__restrict__ thr0, float *__restrict__ sbound) {
  const int b = blockIdx.x, tid = threadIdx.x;
  const float *p = pc + (size_t)b * N * 3;
  float m = 0.f;
  for (int i = tid; i < N; i += 256) {
    const float x = __ldg(p + (size_t)i * 3), y = __ldg(p + (size_t)i * 3 + 1), z = __ldg(p + (size_t)i * 3 + 2);
    m = fmaxf(m, fmaf(z, z, fmaf(y, y, x * x)));
    const float a0 = -2.0f * x, a1 = -2.0f * y, a2 = -2.0f * z, a3 = hg_sumsq3_seq(x, y, z);
    const int *pi = prev + ((size_t)b * N + i) * k1;
    int id[KM];
    float bound = -CUDART_INF_F;
    bool ok = true;
#pragma unroll
    for (int t = 0; t < KM; ++t) {
      id[t] = -1 - t;
      if (t < k1) {
        const int j = __ldg(pi + t);
        id[t] = j;
        if (j < 0 || j >= N) {
          ok = false;
        } else {
          const float cx = __ldg(p + (size_t)j * 3), cy = __ldg(p + (size_t)j * 3 + 1), cz = __ldg(p + (size_t)j * 3 + 2);
          bound = fmaxf(bound, knn_seed_dist(a0, a1, a2, a3, cx, cy, cz, hg_sumsq3_seq(cx, cy, cz)));
        }
      }
    }
#pragma unroll
    for (int t = 1; t < KM; ++t)
#pragma unroll
      for (int u = 0; u < t; ++u) ok = ok && (id[t] != id[u]);
    thr0[(size_t)b * N + i] = ok ? hg_nudge_up(bound) : CUDART_INF_F;
  }
  knn_block_sbound(m, tid, sbound, b);
}

int launch_seed_prev(const float *pc, int B, int N, int k1, const int *prev, float *thr0, float *sbound,
                     cudaStream_t stream) {
  with_km<32>(k1, [&](auto km) {
    knn_seed_prev_kernel<decltype(km)::value><<<B, 256, 0, stream>>>(pc, N, k1, prev, thr0, sbound);
  });
  HG_CHECK_LAUNCH("knn_seed_prev_kernel");
  return HG_OK;
}

// ---- host side of the small-cloud path ---------------------------------------------------------------------
static int g_small_max_n = 0;  // benchmark-only: largest cloud that takes the small-cloud path (0 = default)

template <int QT, int KM, int GP>
int launch_small(const float *pc, int B, int N, int k1, float *vals, int *idx, const float *thr0, const float *sbound,
                 cudaStream_t stream, int *idx_state) {
  const int W = ((N + 1) / 2 + 32 * GP - 1) / (32 * GP);
  if (W > 32) {
    hg_set_error("knn (small-cloud path): N=%d needs %d mask words with GP=%d (max 32)", N, W, GP);
    return HG_E_UNSUPPORTED;
  }
  const size_t smem = (size_t)W * 32 * GP * 2 * sizeof(float4) + (size_t)QT * W * kThreads * sizeof(unsigned);
  if (smem > 48 * 1024)
    HG_CUDA(cudaFuncSetAttribute(knn3_small_kernel<QT, KM, GP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((N + QT * kThreads - 1) / (QT * kThreads), B);
  const bool prof = hg_prof_begin(HG_PROF_KNN, stream);
  knn3_small_kernel<QT, KM, GP><<<grid, kThreads, smem, stream>>>(pc, N, k1, W, vals, idx, thr0, sbound, idx_state);
  hg_prof_end(HG_PROF_KNN, stream, prof);
  HG_CHECK_LAUNCH("knn3_small_kernel");
  return HG_OK;
}

template <int QT, int KM>
int launch_small_gp(int gp, const float *pc, int B, int N, int k1, float *vals, int *idx, const float *thr0,
                    const float *sbound, cudaStream_t stream, int *idx_state) {
  if (gp == 1) return launch_small<QT, KM, 1>(pc, B, N, k1, vals, idx, thr0, sbound, stream, idx_state);
  if (gp == 2) return launch_small<QT, KM, 2>(pc, B, N, k1, vals, idx, thr0, sbound, stream, idx_state);
  return launch_small<QT, KM, 4>(pc, B, N, k1, vals, idx, thr0, sbound, stream, idx_state);
}

int knn3_small_main(const float *pc, int B, int N, int k1, float *vals, int *idx, const float *thr0, const float *sbound,
                    cudaStream_t stream, int *idx_state);

// self-kNN of clouds that fit in shared memory: seeds (one CTA per cloud), then the deferred-drain kernel.
int knn3_small_self(const float *pc, int B, int N, int k1, float *vals, int *idx, float *thr0, float *sbound,
                    cudaStream_t stream, int *idx_state, bool state_valid) {
  if (idx_state && state_valid) {
    int rc = launch_seed_prev(pc, B, N, k1, idx_state, thr0, sbound, stream);
    if (rc) return rc;
    return knn3_small_main(pc, B, N, k1, vals, idx, thr0, sbound, stream, idx_state);
  }
  const size_t seed_smem = (size_t)N * (sizeof(float4) + 2 * sizeof(int));
  // window of the Z-order scan: enough points for a k1-th smallest that is close to the true one
  const int win = k1 <= 8 ? 64 : (k1 <= 16 ? 80 : 96);  // measured (388 x 1024): 64 beats 32 by 5 % at k+1 = 6, 96 beats 64 by 6 % at 20
  const int rc = with_km<32>(k1, [&](auto km) -> int {
    constexpr int kSeedMaxSmem = 8192 * (int)(sizeof(float4) + 2 * sizeof(int));
    static HgPerDeviceOnce once;  // one per instantiation
    if (once.first())
      HG_CUDA(cudaFuncSetAttribute(knn_seed_small_kernel<decltype(km)::value>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   kSeedMaxSmem));
    knn_seed_small_kernel<decltype(km)::value><<<B, 256, seed_smem, stream>>>(pc, N, k1, win, thr0, sbound);
    return HG_OK;
  });
  if (rc) return rc;
  HG_CHECK_LAUNCH("knn_seed_small_kernel");
  return knn3_small_main(pc, B, N, k1, vals, idx, thr0, sbound, stream, idx_state);
}

int knn3_small_main(const float *pc, int B, int N, int k1, float *vals, int *idx, const float *thr0, const float *sbound,
                    cudaStream_t stream, int *idx_state) {
  // Queries per lane / candidate pairs per filter bit (tools/knn_small_sweep.py, B200): two queries per lane amortise
  // the broadcast candidate loads, more would lengthen the serial drains; one pair per bit makes the drain's group
  // re-evaluation cheapest, but needs N/64 mask words per query, which costs occupancy beyond ~1.3k points.
  int gp = g_force_gp ? g_force_gp : (N <= 1280 ? 1 : 2);
  if (N > 2048 && gp < 2) gp = 2;
  if (N > 4096 && gp < 4) gp = 4;
  if (!g_force_gp && k1 > 6 && N > 3072) gp = 4;  // longer lists: 1001 against 1257 us at 64 x 4096, k+1 = 20
  // small batches: one query per lane doubles the CTAs (32 x 1024, k+1 = 6: 51 against 65 us; tools/debug/knn_small_shapes.py)
  // (short candidate lists only: at 16 x 4096 two queries per lane still win, 176 against 212 us); longer lists: one
  int qt = g_force_qt;
  if (!qt)
    qt = (k1 > 6 || (N <= 1536 && (long long)B * ((N + 2 * kThreads - 1) / (2 * kThreads)) < 2LL * hg_sm_count())) ? 1 : 2;
  return with_km_qt<32>(k1, qt, [&](auto km, auto qt_) -> int {
    return launch_small_gp<decltype(qt_)::value, decltype(km)::value>(gp, pc, B, N, k1, vals, idx, thr0, sbound, stream,
                                                                       idx_state);
  });
}

int seed_grid(int N) {
  int G = (int)lroundf(cbrtf((float)N / 3.0f));
  if (G < 1) G = 1;
  if (G > 40) G = 40;
  return G;
}

// 3-D clouds with long neighbour lists (DGCNN layer 1: k = 20) on the tensor-core kernel: the cloud is copied into 32-channel
// rows (x, y, z, 0, ...: a 128-byte row is what the TMA boxes of hg_knn_tc.cu move) and the squared norms are taken with
// the 3-D kernels' operation order.  The zero channels change nothing in the reference's FMA chain (fma(0, 0, acc) = acc),
// so values and indices are the 3-D path's bit for bit.
constexpr int kPadC = 32;
__global__ void __launch_bounds__(256) knn_pad3_kernel(const float *__restrict__ pc, long long total,
                                                       float4 *__restrict__ padded, float *__restrict__ xx) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < total * (kPadC / 4);
       g += (long long)gridDim.x * blockDim.x) {
    const long long row = g / (kPadC / 4);
    const int q = (int)(g - row * (kPadC / 4));
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (q == 0) {
      const float x = __ldg(pc + row * 3), y = __ldg(pc + row * 3 + 1), z = __ldg(pc + row * 3 + 2);
      v = make_float4(x, y, z, 0.f);
      xx[row] = hg_sumsq3_seq(x, y, z);
    }
    padded[g] = v;
  }
}

// shapes that may take the tensor-core kernel on a padded copy (the dispatch also looks at the batch size)
bool knn3_pad_candidate(int N, int k1) { return k1 >= 12 && k1 <= 32 && hg_knn_tc_supported(N, kPadC, k1); }

// Workspace of 3-D self-kNN: the seed area (grid cell of every point; per cloud, stride 8, the grid's origin and scale
// and the bound on max |p|^2; thresholds; cell-sorted points; cell lists), then one region that holds either the padded
// copy for the tensor-core kernel (counted for the shapes that may take it) or the pruned path's kd-tree ordering.
// *_end: the bytes each route needs.
struct Knn3SelfWorkspace {
  int *cellid;
  float *params, *thr0, *padded, *padded_xx;
  float4 *sorted;
  HgSpan cells;
  void *order;
  size_t seed_end, pad_end, order_end;
  Knn3SelfWorkspace(HgCarve &c, int B, int N, int k1) {
    const int G = seed_grid(N);
    cellid = c.take<int>((size_t)B * N);
    params = c.take<float>((size_t)B * 8);
    thr0 = c.take<float>((size_t)B * N);
    sorted = c.take<float4>((size_t)B * N);
    cells = c.span(hg_csr_workspace_bytes(B, G * G * G, N));
    HgCarve pad(c.here()), ord(c.here());
    padded = pad.take<float>((size_t)B * N * kPadC);
    padded_xx = pad.take<float>((size_t)B * N);
    order = ord.span(hg_prune_order_bytes(B, N)).ptr;
    seed_end = c.bytes, pad_end = seed_end + pad.bytes, order_end = seed_end + ord.bytes;
    const size_t shared = knn3_pad_candidate(N, k1) ? pad.bytes : 0;
    c.take<char>(shared > ord.bytes ? shared : ord.bytes);
  }
};

}  // namespace

int hg_knn3_points_i64(const float *p1, const float *p2, int B, int N, int M, int K, float *dists, long long *idx,
                       cudaStream_t stream) {
  return launch_form<HG_KNN_FORM_DIRECT, long long>(p1, p2, B, N, M, K, dists, idx, nullptr, nullptr, stream);
}

size_t hg_knn3_self_workspace_bytes(int B, int N, int k1) { return hg_layout_bytes<Knn3SelfWorkspace>(B, N, k1); }

// Benchmark-only overrides: the smallest cloud that gets grid-seeded thresholds (0 = default) and the seed scan's
// neighbourhood (0 = automatic, 1 = 2x2x2 cells, 2 = 3x3x3 cells).
static int g_seed_min_n = 0, g_seed_near8 = 0;
HG_API void hg_knn_tune(int seed_min_n, int near8) {
  g_seed_min_n = seed_min_n;
  g_seed_near8 = near8;
}

HG_API void hg_knn_force_shape(int qt, int gp) {
  g_force_qt = qt;
  g_force_gp = gp;
}

HG_API void hg_knn_tune_small(int small_max_n) { g_small_max_n = small_max_n; }

// Self-kNN (expanded form) of 3-D clouds.  Routes by precedence: pruned search, tensor-core kernel on a padded copy,
// unseeded all-pairs kernel, small-cloud kernel, then the streaming kernel with the 4-operation folded filter seeded
// from the previous call's neighbours, from a bound alone or from the grid pre-pass.
// idx_state (optional, [B,N,k1]): the neighbour indices of the previous call on a nearby cloud -- read as temporal
// seeds when state_valid, and overwritten with this call's indices (a second copy of idx).
int hg_knn3_self_i32(const float *pc, int B, int N, int k1, float *vals, int *idx, int *idx_state, int state_valid,
                     void *order, void *workspace, size_t workspace_bytes, cudaStream_t stream) {
  const auto w = hg_layout_at<Knn3SelfWorkspace>(workspace, B, N, k1);
  if (hg_prune_applies(N) && workspace != nullptr && workspace_bytes >= w.order_end) {
    // large clouds: kd-tree ordering and pruned search (hg_prune.cu), seeded from each query's own leaf or, with
    // temporal seeds, from the previous call's neighbours; clouds the ordering flags (non-finite coordinates) then
    // take the all-pairs kernel with the reference arithmetic
    const float *thr0 = nullptr;
    if (idx_state && state_valid && k1 <= 32) {  // (the seed kernel bounds at most 32 previous neighbours)
      int rc = launch_seed_prev(pc, B, N, k1, idx_state, w.thr0, w.params, stream);
      if (rc) return rc;
      thr0 = w.thr0;
    }
    HgPruneOrder o;
    const bool prof = hg_prof_begin(HG_PROF_KNN, stream);
    int rc = hg_prune_build(pc, B, N, false, w.order, &o, stream, order);
    if (!rc) rc = hg_prune_knn_search(o, B, k1, thr0, vals, idx, idx_state, stream);
    hg_prof_end(HG_PROF_KNN, stream, prof);
    if (rc) return rc;
    return launch_form<HG_KNN_FORM_EXPANDED, int>(pc, pc, B, N, N, k1, vals, idx, nullptr, nullptr, stream, idx_state,
                                                  o.info);
  }
  // long lists on enough clouds to fill the machine: the tensor-core kernel on a 32-channel copy beats the 3-D
  // small-cloud kernel up to ~8 CTAs per SM (k = 20, 1024 points: 16 clouds 62 against 131 us, 32: 78 / 136, 128: 221 / 236,
  // 192: 326 / 313; 2048 points: 32 clouds 196 / 244, 96: 485 / 464); KNNDist's short lists (and its temporal state) stay 3-D
  if (!hg_prune_applies(N) && !idx_state && knn3_pad_candidate(N, k1) && g_hg_tune_knn_tc_off != 1 && workspace &&
      workspace_bytes >= w.pad_end &&
      ((4LL * B * ((N + 127) / 128) >= hg_sm_count() && (long long)B * ((N + 127) / 128) <= 8LL * hg_sm_count()) ||
       g_hg_tune_knn_tc_off == 2 || g_hg_tune_knn_tc_off == 5)) {
    const long long rows = (long long)B * N;
    knn_pad3_kernel<<<hg_grid_for(rows * (kPadC / 4), 256, 16), 256, 0, stream>>>(pc, rows, (float4 *)w.padded, w.padded_xx);
    HG_CHECK_LAUNCH("knn_pad3_kernel");
    return hg_knn_tc_run(w.padded, w.padded_xx, B, N, kPadC, k1, vals, idx, stream);
  }
  if (k1 > 32 || workspace == nullptr || workspace_bytes < w.seed_end)
    return launch_form<HG_KNN_FORM_EXPANDED, int>(pc, pc, B, N, N, k1, vals, idx, nullptr, nullptr, stream, idx_state);
  // (tools/debug/knn_mid_sweep.py, B200, k+1 = 6: 2048 points 209 against 311 us streaming, 3000: 317 / 403, 4096: 444 / 458,
  // 8192: 1237 / 688)
  const int small_max = g_small_max_n > 0 ? (g_small_max_n < 8192 ? g_small_max_n : 8192) : (g_small_max_n < 0 ? -1 : 4096);
  if (N <= small_max)  // clouds that fit in shared memory: deferred-drain kernel
    return knn3_small_self(pc, B, N, k1, vals, idx, w.thr0, w.params, stream, idx_state, state_valid != 0);
  if (idx_state && state_valid) {  // temporal seeds instead of the grid pre-pass
    int rc = launch_seed_prev(pc, B, N, k1, idx_state, w.thr0, w.params, stream);
    if (rc) return rc;
    return launch_form<HG_KNN_FORM_EXPANDED_FOLD4, int>(pc, pc, B, N, N, k1, vals, idx, w.thr0, w.params, stream, idx_state);
  }
  if (N < (g_seed_min_n > 0 ? g_seed_min_n : 2048)) {
    // (benchmark-only, when the small-cloud path is switched off) cold thresholds with the 4-operation folded filter
    knn_bound_kernel<<<B, 256, 0, stream>>>(pc, N, w.params);
    HG_CHECK_LAUNCH("knn_bound_kernel");
    return launch_form<HG_KNN_FORM_EXPANDED_FOLD4, int>(pc, pc, B, N, N, k1, vals, idx, nullptr, w.params, stream, idx_state);
  }
  const int G = seed_grid(N), ncell = G * G * G;
  knn_cells_kernel<<<B, 256, 0, stream>>>(pc, N, G, w.cellid, w.params);
  HG_CHECK_LAUNCH("knn_cells_kernel");
  HgCsr csr;
  int rc = hg_csr_build_unordered(w.cellid, B, N, ncell, w.cells.ptr, w.cells.bytes, &csr, stream);
  if (rc) return rc;
  knn_cell_sort_kernel<<<hg_grid_for((long long)B * N, 256, 16), 256, 0, stream>>>(pc, csr.list, (long long)B * N, N,
                                                                                     w.sorted);
  HG_CHECK_LAUNCH("knn_cell_sort_kernel");
  dim3 grid((N + 127) / 128, B);
  // neighbourhood of the seed scan: the 2x2x2 cells nearest to the query (3.4x fewer candidates, a slightly looser
  // bound: measured 5-9 % faster end to end at k+1 = 6, 2-5 % at k+1 = 20), all 27 cells for longer lists, which the
  // ~24 points of 8 cells cannot fill (tools/knn_seed_sweep.py)
  const int near8 = g_seed_near8 == 1 ? 1 : g_seed_near8 == 2 ? 0 : (k1 <= 20);
  with_km<32>(k1, [&](auto km) {
    knn_seed_kernel<decltype(km)::value><<<grid, 128, 0, stream>>>(w.sorted, N, G, w.params, csr.off, csr.list, w.thr0,
                                                                   near8);
  });
  HG_CHECK_LAUNCH("knn_seed_kernel");
  // seeded path: the bounding box is known, so the main loop can run the 4-operation folded filter
  return launch_form<HG_KNN_FORM_EXPANDED_FOLD4, int>(pc, pc, B, N, N, k1, vals, idx, w.thr0, w.params + 6, stream, idx_state);
}
