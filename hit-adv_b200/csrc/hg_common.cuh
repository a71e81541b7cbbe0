// hg_common.cuh -- shared helpers of libhitgeom (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/hitgeom.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libhitgeom is written for sm_100a (B200) only"
#endif

#define HG_API extern "C" __attribute__((visibility("default")))

// ---- error reporting (thread-local message, never exit()) -------------------------------------------------
void hg_set_error(const char *fmt, ...);

#define HG_REQUIRE(cond, code, ...)   \
  do {                                \
    if (!(cond)) {                    \
      hg_set_error(__VA_ARGS__);      \
      return (code);                  \
    }                                 \
  } while (0)

// NVTX range around every compute entry point of the C ABI (header-only NVTX v3: a no-op unless a tool is attached),
// so that nsys / ncu timelines of a reference run show which reference call a kernel belongs to
struct HgNvtxRange {
  explicit HgNvtxRange(const char *name) { nvtxRangePushA(name); }
  ~HgNvtxRange() { nvtxRangePop(); }
  HgNvtxRange(const HgNvtxRange &) = delete;
  HgNvtxRange &operator=(const HgNvtxRange &) = delete;
};
#define HG_NVTX_RANGE(name) HgNvtxRange hg_nvtx_range_(name)

extern int g_hg_tune_knn_tc_off;  // hg_tune("knn_tc", 1) switches the tensor-core kNN prefilter off
extern int g_hg_tune_small_fused_off;  // hg_tune("small_fused", 1): general paths for small clouds too (A/B, tests)
extern unsigned long long g_hg_launches;  // kernels launched by this library (bench.py's gpu_launches)

#define HG_CHECK_LAUNCH(name)                                            \
  do {                                                                   \
    ++g_hg_launches;                                                     \
    cudaError_t e__ = cudaGetLastError();                                \
    if (e__ != cudaSuccess) {                                            \
      hg_set_error("%s: %s", (name), cudaGetErrorString(e__));           \
      return (int)e__;                                                   \
    }                                                                    \
  } while (0)

#define HG_CUDA(call)                                                    \
  do {                                                                   \
    cudaError_t e__ = (call);                                            \
    if (e__ != cudaSuccess) {                                            \
      hg_set_error("%s: %s", #call, cudaGetErrorString(e__));            \
      return (int)e__;                                                   \
    }                                                                    \
  } while (0)

static inline cudaStream_t hg_stream(hgStream s) { return reinterpret_cast<cudaStream_t>(s); }

static inline size_t hg_align(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// A workspace layout is written once, as a type constructed from (HgCarve &, arguments): take() hands out the next
// region, rounded up to 256 bytes.  On a null base it only counts: hg_layout_bytes is the size, hg_layout_at the pointers.
struct HgSpan { void *ptr; size_t bytes; };  // a region that a callee carves itself
struct HgCarve {
  char *base;
  size_t bytes = 0;
  explicit HgCarve(void *base_ = nullptr) : base((char *)base_) {}
  char *here() const { return base ? base + bytes : nullptr; }
  template <typename T> T *take(size_t n) { T *p = (T *)here(); bytes += hg_align(n * sizeof(T)); return p; }
  HgSpan span(size_t n) { return {take<char>(n), hg_align(n)}; }
};
template <typename Layout, typename... A> size_t hg_layout_bytes(A... a) { HgCarve c; Layout(c, a...); return c.bytes; }
template <typename Layout, typename... A> Layout hg_layout_at(void *base, A... a) { HgCarve c(base); return Layout(c, a...); }

int hg_sm_count();
// blocks of `threads` for a grid-stride loop over `total` items: enough to cover them, at most per_sm per SM, at least one
static inline int hg_grid_for(long long total, int threads, int per_sm) {
  long long blocks = (total + threads - 1) / threads;
  const long long cap = (long long)hg_sm_count() * per_sm;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}
// true the first time it is called on the current device with this flag array (function attributes such as the
// dynamic shared-memory limit are per device: one `static` flag per process would miss the second GPU)
struct HgPerDeviceOnce {
  unsigned char done[64] = {0};
  bool first() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    if (done[dev]) return false;
    done[dev] = 1;
    return true;
  }
};

// per-kernel device timing hooks (hg_abi.cu); tags are part of the ABI (include/hitgeom.h HG_PROF_*)
bool hg_prof_begin(int tag, cudaStream_t s);
void hg_prof_end(int tag, cudaStream_t s, bool began);

// ---- exact FP32 building blocks (SURVEY.md section 8 a-bis) ------------------------------------------------
// Everything that decides an index goes through these intrinsics, which nvcc never contracts or reorders.

// torch.bmm with inner dim 3: fma(a2,b2, fma(a1,b1, a0*b0))
__device__ __forceinline__ float hg_dot3_fma(float a0, float a1, float a2, float b0, float b1, float b2) {
  return __fmaf_rn(a2, b2, __fmaf_rn(a1, b1, __fmul_rn(a0, b0)));
}
// torch.sum(x**2, dim) for three channels: (a0*a0 + a1*a1) + a2*a2, no FMA
__device__ __forceinline__ float hg_sumsq3_seq(float a0, float a1, float a2) {
  return __fadd_rn(__fadd_rn(__fmul_rn(a0, a0), __fmul_rn(a1, a1)), __fmul_rn(a2, a2));
}
// nvcc -O3 contraction of (ax-bx)*(ax-bx) + (ay-by)*(ay-by) + (az-bz)*(az-bz) in the pointnet2_ops kernels:
// fma(dz,dz, fma(dx,dx, round(dy*dy))) -- in `a*a + b*b` the LEFT product is fused, the right one rounded (read
// off the SASS of query_ball_point_kernel / three_nn_kernel / furthest_point_sampling_kernel built for sm_100).
__device__ __forceinline__ float hg_dist3_fma(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}
// pytorch3d knn_points: `dist += diff*diff` per coordinate -> fma(dz,dz, fma(dy,dy, dx*dx))
__device__ __forceinline__ float hg_dist3_seq(float ax, float ay, float az, float bx, float by, float bz) {
  const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
  return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}

// order-preserving float <-> uint32 (so that integer min/max atomics select the float min/max exactly)
__device__ __forceinline__ unsigned hg_ord(float f) {
  const unsigned u = __float_as_uint(f);
  return u ^ (((unsigned)((int)u >> 31)) | 0x80000000u);
}
__device__ __forceinline__ float hg_unord(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
}

// d into the ascending list v of the KM smallest values so far, without branches: each level keeps the smaller and passes
// the larger on.  fminf / fmaxf drop a NaN d, and the level then duplicates its entry: keep NaN out of d.
template <int KM>
__device__ __forceinline__ void hg_sorted_min_insert(float (&v)[KM], float d) {
#pragma unroll
  for (int u = 0; u < KM; ++u) {
    const float lo = fminf(v[u], d);
    d = fmaxf(v[u], d);
    v[u] = lo;
  }
}

// the next float above v (+inf for +inf and NaN): turns a bound that a strict '<' filter tests into one that keeps ties
__device__ __forceinline__ float hg_nudge_up(float v) {
  return v < CUDART_INF_F ? nextafterf(v, CUDART_INF_F) : CUDART_INF_F;
}

__device__ __forceinline__ float hg_warp_min_f32(float v) {
  float m;
  asm("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));  // CREDUX.MIN.F32 (sm_100a)
  return m;
}
__device__ __forceinline__ float hg_warp_max_f32(float v) {
  float m;
  asm("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(v));
  return m;
}

// ---- bulk asynchronous copies (TMA unit, 1-D): global -> shared, completion on an mbarrier ------------------------
// cp.async.bulk (SASS: UBLKCP) moves a whole contiguous block with ONE instruction issued by one thread; the copy
// engine keeps it in flight while the CTA computes on the previous block.  Sizes and both addresses must be multiples
// of 16 bytes.  hg_mbar_wait spins on the phase parity (try_wait suspends the thread in hardware between polls).
__device__ __forceinline__ unsigned hg_smem_addr(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void hg_mbar_init(uint64_t *bar, unsigned arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(hg_smem_addr(bar)), "r"(arrivals) : "memory");
}
__device__ __forceinline__ void hg_mbar_init_fence() {  // make the initialised barriers visible to the async proxy
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void hg_mbar_expect_tx(uint64_t *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(hg_smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hg_bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   hg_smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(hg_smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void hg_mbar_wait(uint64_t *bar, unsigned parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "HG_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra HG_DONE_%=;\n\t"
      "bra HG_WAIT_%=;\n\t"
      "HG_DONE_%=:\n\t"
      "}" ::"r"(hg_smem_addr(bar)),
      "r"(parity)
      : "memory");
}

// __match_any_sync on keys of `nbits` bits, built from ballots: MATCH.ANY resolves one distinct value at a time (about
// 600 cycles for 32 distinct keys, measured through the CSR builder: 48 us for 16k edges per cloud), a ballot per key
// bit costs a few cycles each
__device__ __forceinline__ unsigned hg_match_any_bits(int key, int nbits) {
  unsigned same = 0xffffffffu;
  for (int b = 0; b < nbits; ++b) {
    const bool bit = (key >> b) & 1;
    const unsigned v = __ballot_sync(0xffffffffu, bit);
    same &= bit ? v : ~v;
  }
  return same;
}

// ---- deterministic reverse map (CSR) used by every scatter-style backward ----------------------------------
// keys [B,E] (destination of edge e, or <0 to skip) -> off [B,N+1], list [B,E] with, for each destination,
// its edges in ascending e.  Summing in list order is what replaces the reference's float atomicAdd.
size_t hg_csr_workspace_bytes(int B, int N, int E);         // for hg_csr_build_unordered
size_t hg_csr_stable_workspace_bytes(int B, int N, int E);  // for hg_csr_build
struct HgCsr {
  int *off;   // [B, N+1]
  int *list;  // [B, E]
};
int hg_csr_build(const int *keys, int B, int E, int N, void *workspace, size_t workspace_bytes, HgCsr *out,
                 cudaStream_t stream);
// Same layout, built with parallel integer atomics: entries of a segment are in arbitrary order, walk them with
// hg_csr_next() to get ascending edge order (deterministic sums without a stable sort).
int hg_csr_build_unordered(const int *keys, int B, int E, int N, void *workspace, size_t workspace_bytes, HgCsr *out,
                           cudaStream_t stream);
// workspace of a scatter-style backward: keys [B,E], then the CSR build (stable or unordered) that groups them
struct HgKeysCsr {
  int *keys;
  HgSpan csr;
  HgKeysCsr(HgCarve &c, int B, int N, long long E, bool stable)
      : keys(c.take<int>((size_t)B * E)),
        csr(c.span(stable ? hg_csr_stable_workspace_bytes(B, N, (int)E) : hg_csr_workspace_bytes(B, N, (int)E))) {}
};
// smallest entry of list[p0..p1) that is greater than `last` (INT_MAX if none)
__device__ __forceinline__ int hg_csr_next(const int *__restrict__ list, int p0, int p1, int last) {
  int best = 0x7fffffff;
  for (int q = p0; q < p1; ++q) {
    const int e = list[q];
    if (e > last && e < best) best = e;
  }
  return best;
}

// ---- tensor-core kNN prefilter for feature clouds (hg_knn_tc.cu) ---------------------------------------------------
bool hg_knn_tc_supported(int K, int C, int k1);
bool hg_knn_tc_supported_feature(int K, int C, int k1);
int hg_knn_tc_run(const float *pc, const float *xx, int B, int K, int C, int k1, float *vals, int *idx, cudaStream_t stream);

// ---- spatially pruned exact passes for large clouds (hg_prune.cu) ---------------------------------------------------
#define HG_PRUNE_MAX_N 16384  // the ordering build holds one cloud in shared memory and keys with 14-bit point indices
// One cloud batch in kd-tree order: points (x, y, z, squared norm), original index of every sorted point, per-leaf
// boxes (lo, hi) of 32 points, per-cloud (bound on max |p|^2, 1 if the cloud must take the all-pairs kernels).
struct HgPruneOrder {
  float4 *pts;   // [B,N]
  int *perm;     // [B,N]
  float4 *box;   // [B,ceil(N/32),2]
  float4 *info;  // [B]
  int N;
};
int hg_prune_tune(const char *key, int value);  // 1 if the key is one of the pruned path's
bool hg_prune_applies(int N);               // the size threshold and hg_tune("prune") as they stand
size_t hg_prune_order_bytes(int B, int N);  // 0 when the path does not apply to N
// state (null, or an ordering state of hg_order_state_bytes(B, N) bytes): refit the state's permutation and rebuild only
// the clouds whose refit fails (hg_prune.cu); o->perm then points into the state
int hg_prune_build(const float *pc, int B, int N, bool chamfer_norm, void *ws, HgPruneOrder *o, cudaStream_t stream,
                   void *state = nullptr);
int hg_prune_nn_search(const HgPruneOrder &q, const HgPruneOrder &c, int B, float *mins, int *args, cudaStream_t stream);
int hg_prune_knn_search(const HgPruneOrder &o, int B, int k1, const float *thr0, float *vals, int *idx, int *idx_state,
                        cudaStream_t stream);

// ---- 3-D streaming kNN (hg_knn3.cu) ---------------------------------------------------------------------------
// pytorch3d knn_points: the K nearest of p2 to every point of p1, with its arithmetic (arguments checked by the caller)
int hg_knn3_points_i64(const float *p1, const float *p2, int B, int N, int M, int K, float *dists, long long *idx,
                       cudaStream_t stream);
// 3-D self-kNN (expanded form), every route: hg_knn_self_temporal_order_f32 with C = 3 (arguments checked there)
size_t hg_knn3_self_workspace_bytes(int B, int N, int k1);
int hg_knn3_self_i32(const float *pc, int B, int N, int k1, float *vals, int *idx, int *idx_state, int state_valid,
                     void *order, void *workspace, size_t workspace_bytes, cudaStream_t stream);
