// hg_knn_tc.cu -- k-nearest-neighbour search on FEATURE clouds (DGCNN edge-conv layers 2-4: C = 64, 64, 128 channels,
// model/dgcnn_cls.py:7-13): a tensor-core filter fused with the exact FP32 evaluation of what it lets through.
//
// The distance matrix of a C-channel cloud is a real contraction (2*C FLOP per pair), the one place on this path where
// the 5th-generation tensor cores are admissible (SURVEY.md section 8d) -- provided every index stays the reference's.
// Tensor cores multiply in TF32, so their distances only SELECT candidates; every value and index that is returned
// comes from the reference's FP32 arithmetic:
//
//   knn_tc_fused_kernel (tcgen05 + TMEM + TMA).  One CTA per (cloud, 128 query rows).  The 128 x C query block and the
//   256 x C candidate tiles (both K-major slices of the same [K, C] matrix) are brought in by TMA (cp.async.bulk.tensor,
//   128-byte swizzle) and multiplied with tcgen05.mma.kind::tf32 into a 128 x 256 FP32 accumulator in tensor memory; the
//   four warps read it back with tcgen05.ld (thread = row) and turn it into a hit mask: columns whose approximate
//   distance is <= threshold + 2 eps, where eps bounds |approximate - reference| for that row: TF32 keeps 11 significant
//   bits of each operand, so |zz_tf32 - zz| <= |x_i||x_j| 2^-9 and eps_i = 1.1 * 2^-8 |x_i| max|x| + (FP32 rounding of
//   both sides).  Every hit is evaluated EXACTLY on the spot, out of the same shared-memory tile (see the kernel's comment).
// Nothing of size K x K is stored, and no candidate list leaves the SM.
//
// History (round 2): a two-kernel version -- two-pass filter writing candidate lists, then a warp-per-row exact kernel
// gathering the candidates' rows from L2 -- took 163 us at 32 x 1024 x 64 (filter 50 us, gather-bound exact kernel 88 us);
// the fused pass takes 99 us for the whole call (75 us the kernel; 130 us with a single sweep, see two_pass).  A variant
// with two threads per row (16 warps per SM, two partial lists merged at the end) was slower (156 us against 135): the exact phase is bound by shared-memory bandwidth (random candidate rows:
// 1.9 wavefronts per ideal one), not by latency, and two lists admit more candidates than one.
#include <cuda.h>

#include "hg_common.cuh"

namespace {

constexpr int kTcRows = 128;    // query rows per CTA (UMMA M)
constexpr int kTcTile = 256;    // candidate columns per accumulator tile (UMMA N)
constexpr int kTcPanelK = 32;   // TF32 elements per 128-byte swizzled panel row

// ---- small PTX wrappers (tcgen05 / TMA / mbarrier) ----------------------------------------------------------------
__device__ __forceinline__ void tc_mbar_wait(uint64_t *bar, unsigned parity) {
  // bounded spin: a protocol bug must surface as a trapped kernel, never as a hung GPU
  unsigned ok = 0;
  for (unsigned spin = 0; spin < (1u << 28); ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(hg_smem_addr(bar)), "r"(parity)
        : "memory");
    if (ok) return;
  }
  __trap();
}
__device__ __forceinline__ void tc_tma_load_3d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          hg_smem_addr(dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(hg_smem_addr(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(hg_smem_addr(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// shared-memory matrix descriptor of a K-major, 128-byte-swizzled panel ([rows] x 128 bytes, 8-row groups 1024 bytes
// apart): start address, LBO = 1 (unused for swizzled K-major), SBO = 1024 B, version 1 (Blackwell), SWIZZLE_128B
__device__ __forceinline__ uint64_t tc_smem_desc(const void *panel, int k_byte_offset) {
  const uint32_t addr = hg_smem_addr(panel) + (uint32_t)k_byte_offset;
  uint64_t d = 0;
  d |= (uint64_t)((addr & 0x3FFFFu) >> 4);        // bits [0,14)
  d |= (uint64_t)1 << 16;                         // leading byte offset (>>4) = 1
  d |= (uint64_t)(1024 >> 4) << 32;               // stride byte offset (>>4)
  d |= (uint64_t)1 << 46;                         // descriptor version
  d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
  return d;
}
// instruction descriptor: D = F32, A = B = TF32, both K-major, M = 128, N = 256
__host__ __device__ constexpr uint32_t tc_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// Column norms.  Up to 4096 points (kTileNorms = false) the norms of the whole cloud stay resident in shared memory,
// ceil(K/256) * 1 KiB.  Beyond that (kTileNorms = true, up to 16384 points) only the current candidate tile's 256 norms
// are: every thread loads two of them from global memory (L2) while the tile's TMA loads and MMAs are in flight, and
// one barrier after those completes makes them visible to the CTA.  The B panels are single-buffered (the next tile is
// loaded only once every warp has released the current one), so one 1 KiB slot is enough, and shared memory no longer
// depends on K.  (Not a cp.async.bulk on the tile's mbarrier: a cloud's norms start at b * K floats, 16-byte
// aligned only when K % 4 == 0.)  max|x|, the error bound's cloud term, is still taken over all K rows.
__device__ __forceinline__ void tc_stage_tile_norms(float *slot, const float *xxb, int K, int t, int tid) {
  const int j0 = t * kTcTile + tid, j1 = j0 + 128;
  slot[tid] = j0 < K ? xxb[j0] : CUDART_INF_F;
  slot[tid + 128] = j1 < K ? xxb[j1] : CUDART_INF_F;
}

// ---- fused single pass: tensor-core filter + exact FP32 evaluation out of the SAME shared-memory tiles --------------
// The candidate tile that TMA brought in for the MMA holds, row by row, exactly the FP32 features the reference
// arithmetic needs.  So a column the TF32 distances cannot rule out is evaluated on the spot -- the thread (= query row)
// keeps its own row in registers (C <= 64) or re-reads it from the A panels, walks the candidate's 128-byte-swizzled row
// with conflict-free 16-byte loads, runs the reference's sequential FMA chain and inserts (value, index) into a sorted
// register list of the row's KM smallest.  Columns are visited in ascending order, so a strict '<' insertion keeps the
// lowest index among equal values (torch.topk's order on this path, hg_knn.cu).  The admission threshold starts from
// the k-th smallest of 32 column-class minima (an upper bound on the k-th smallest approximate distance) -- taken over
// ALL columns by a first, MMA-only sweep (two_pass, the default), or over tile 0 only -- and follows the list's k-th
// EXACT value from then on:  approx_j <= (k-th exact so far) + 2 eps  is necessary for column j to enter the final
// list, eps bounding |approximate - reference| for the row (header).  The first sweep costs a second round of TMA loads
// and MMAs and halves the exact evaluations (130 -> 99 us).  No candidate lists in global memory, no L2 gathers.
template <int KM>
struct TcList {
  float v[KM];
  int id[KM];
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int s = 0; s < KM; ++s) {
      v[s] = CUDART_INF_F;
      id[s] = 0;
    }
  }
  // sorted insertion, strict '<': an equal value stays behind the entries already there
  __device__ __forceinline__ void push(float d, int j) {
#pragma unroll
    for (int s = KM - 1; s >= 1; --s) {
      const bool above = d < v[s - 1], here = d < v[s];
      id[s] = above ? id[s - 1] : (here ? j : id[s]);
      v[s] = above ? v[s - 1] : (here ? d : v[s]);
    }
    if (d < v[0]) {
      v[0] = d;
      id[0] = j;
    }
  }
  // k1-th smallest = maximum of the first k1 entries of the ascending list (written as a masked maximum: a
  // "select entry k1-1" chain is turned into a dynamically indexed load by the compiler, which sends the list to local memory)
  __device__ __forceinline__ float kth(int k1) const {
    float r = -CUDART_INF_F;
#pragma unroll
    for (int s = 0; s < KM; ++s)
      if (s < k1) r = fmaxf(r, v[s]);
    return r;
  }
};

template <int C, int KM, bool kTileNorms>
__global__ void __launch_bounds__(128, C <= 64 ? 2 : 1)
    knn_tc_fused_kernel(const __grid_constant__ CUtensorMap map, int K, int k1, int two_pass,
                        const float *__restrict__ xx, float *__restrict__ vals, int *__restrict__ idx) {
  constexpr int NP = C / kTcPanelK;
  constexpr int kABytes = kTcRows * 128, kBBytes = kTcTile * 128;
  constexpr bool kOwnInRegs = C <= 64;
  extern __shared__ __align__(1024) unsigned char smraw[];
  unsigned char *sA = smraw, *sB = smraw + NP * kABytes;
  float *sxx = reinterpret_cast<float *>(sB + NP * kBBytes);
  __shared__ __align__(8) uint64_t bar_a, bar_b, bar_mma;
  __shared__ uint32_t tmem_base_s;
  __shared__ float wmax[4];

  const int b = blockIdx.y, row0 = blockIdx.x * kTcRows;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int ntiles = (K + kTcTile - 1) / kTcTile;

  if (tid == 0) {
    hg_mbar_init(&bar_a, 1);
    hg_mbar_init(&bar_b, 1);
    hg_mbar_init(&bar_mma, 1);
    hg_mbar_init_fence();
  }
  if (warp == 0) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(hg_smem_addr(&tmem_base_s))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  float xmax = 0.f;  // largest squared norm of the cloud (for the error bound below)
  if (kTileNorms) {
    for (int j = tid; j < K; j += 128) xmax = fmaxf(xmax, xx[(size_t)b * K + j]);
  } else {
    for (int j = tid; j < ntiles * kTcTile; j += 128) {
      const float v = j < K ? xx[(size_t)b * K + j] : CUDART_INF_F;
      sxx[j] = v;
      if (j < K) xmax = fmaxf(xmax, v);
    }
  }
  xmax = hg_warp_max_f32(xmax);
  if ((tid & 31) == 0) wmax[warp] = xmax;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  xmax = fmaxf(fmaxf(wmax[0], wmax[1]), fmaxf(wmax[2], wmax[3]));

  if (tid == 0) {
    hg_mbar_expect_tx(&bar_a, NP * kABytes);
    for (int p = 0; p < NP; ++p) tc_tma_load_3d(sA + p * kABytes, &map, &bar_a, p * kTcPanelK, row0, b);
  }

  const int i = row0 + tid;
  const bool live = i < K;
  const float xi = live ? (kTileNorms ? xx[(size_t)b * K + i] : sxx[i]) : 0.f;
  const float eps = 1.1f * 0.00390625f * sqrtf(xi * xmax) + 1e-5f * (xi + xmax);
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const unsigned sw = (unsigned)(tid & 7);  // swizzle phase of this thread's own row in the A panels

  float4 own[kOwnInRegs ? C / 4 : 1];
  TcList<KM> top;
  top.init();
  float thr = CUDART_INF_F;
  unsigned phase_b = 0, phase_m = 0;

  // reference distances of columns jr0, jr1 of the current tile (two independent chains in flight): zz = sequential
  // FMA chain over the channels in ascending order, dist = (xx_j + (-2 zz)) + xx_i; + 0.0f turns a -0.0 into +0.0 like
  // the selection kernels do
  auto exact2 = [&](int jr0, int jr1, float xxj0, float xxj1, float &d0, float &d1) {
    float acc0 = 0.f, acc1 = 0.f;
    const unsigned sw0 = (unsigned)(jr0 & 7), sw1 = (unsigned)(jr1 & 7);
#pragma unroll
    for (int p = 0; p < NP; ++p) {
      const unsigned char *r0 = sB + p * kBBytes + jr0 * 128, *r1 = sB + p * kBBytes + jr1 * 128;
      const unsigned char *rowi = sA + p * kABytes + tid * 128;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float4 v0 = *reinterpret_cast<const float4 *>(r0 + ((c ^ sw0) << 4));
        const float4 v1 = *reinterpret_cast<const float4 *>(r1 + ((c ^ sw1) << 4));
        const float4 a = kOwnInRegs ? own[kOwnInRegs ? p * 8 + c : 0]
                                    : *reinterpret_cast<const float4 *>(rowi + ((c ^ sw) << 4));
        acc0 = __fmaf_rn(a.x, v0.x, acc0);
        acc1 = __fmaf_rn(a.x, v1.x, acc1);
        acc0 = __fmaf_rn(a.y, v0.y, acc0);
        acc1 = __fmaf_rn(a.y, v1.y, acc1);
        acc0 = __fmaf_rn(a.z, v0.z, acc0);
        acc1 = __fmaf_rn(a.z, v1.z, acc1);
        acc0 = __fmaf_rn(a.w, v0.w, acc0);
        acc1 = __fmaf_rn(a.w, v1.w, acc1);
      }
    }
    d0 = __fadd_rn(__fadd_rn(__fadd_rn(xxj0, __fmul_rn(-2.0f, acc0)), xi), 0.0f);
    d1 = __fadd_rn(__fadd_rn(__fadd_rn(xxj1, __fmul_rn(-2.0f, acc1)), xi), 0.0f);
  };

  // two_pass: a first, MMA-only sweep over all tiles gives the threshold from the class minima of ALL columns (about
  // half the exact evaluations of the single sweep, for a second round of TMA loads and MMAs)
  float m[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) m[c] = CUDART_INF_F;
  const int nsteps = two_pass ? 2 * ntiles : ntiles;
  for (int step = 0; step < nsteps; ++step) {
    const int t = step < ntiles ? step : step - ntiles;
    const bool scan = two_pass ? step < ntiles : step == 0;       // class minima of this tile
    const bool last_scan = two_pass ? step == ntiles - 1 : step == 0;
    const bool eval = !two_pass || step >= ntiles;                // hits of this tile, evaluated exactly
    if (tid == 0) {
      hg_mbar_expect_tx(&bar_b, NP * kBBytes);
      for (int p = 0; p < NP; ++p) {
        tc_tma_load_3d(sB + p * kBBytes, &map, &bar_b, p * kTcPanelK, t * kTcTile, b);
        tc_tma_load_3d(sB + p * kBBytes + kABytes, &map, &bar_b, p * kTcPanelK, t * kTcTile + 128, b);
      }
      if (step == 0) tc_mbar_wait(&bar_a, 0);
      tc_mbar_wait(&bar_b, phase_b);
      tc_fence_after();
      constexpr uint32_t idesc = tc_idesc(kTcRows, kTcTile);
#pragma unroll
      for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          tc_mma_tf32(tmem, tc_smem_desc(sA + p * kABytes, ks * 32), tc_smem_desc(sB + p * kBBytes, ks * 32), idesc,
                      (p | ks) ? 1u : 0u);
      tc_commit(&bar_mma);
    }
    if (kTileNorms) tc_stage_tile_norms(sxx, xx + (size_t)b * K, K, t, tid);
    // every thread reads the tiles with ordinary loads below: each one observes the TMA completions itself
    if (step == 0) {
      tc_mbar_wait(&bar_a, 0);
      if (kOwnInRegs) {
#pragma unroll
        for (int p = 0; p < NP; ++p)
#pragma unroll
          for (int c = 0; c < 8; ++c)
            own[kOwnInRegs ? p * 8 + c : 0] =
                *reinterpret_cast<const float4 *>(sA + p * kABytes + tid * 128 + ((c ^ sw) << 4));
      }
    }
    tc_mbar_wait(&bar_b, phase_b);
    phase_b ^= 1;
    tc_mbar_wait(&bar_mma, phase_m);
    phase_m ^= 1;
    __syncwarp();
    tc_fence_after();
    if (kTileNorms) __syncthreads();  // the tile's norms, stored by all four warps

    if (scan) {
      // first threshold: k1-th smallest of the 32 column-class minima of the approximate distances scanned so far
#pragma unroll 1
      for (int q = 0; q < kTcTile / 32; ++q) {
        float acc[32];
        tc_ld32(trow + (uint32_t)(q * 32), acc);
        const float4 *sx4 = reinterpret_cast<const float4 *>(kTileNorms ? sxx + q * 32 : sxx + t * kTcTile + q * 32);
#pragma unroll
        for (int c4 = 0; c4 < 8; ++c4) {
          const float4 xj = sx4[c4];
          m[4 * c4] = fminf(m[4 * c4], fmaf(-2.0f, acc[4 * c4], xi + xj.x));
          m[4 * c4 + 1] = fminf(m[4 * c4 + 1], fmaf(-2.0f, acc[4 * c4 + 1], xi + xj.y));
          m[4 * c4 + 2] = fminf(m[4 * c4 + 2], fmaf(-2.0f, acc[4 * c4 + 2], xi + xj.z));
          m[4 * c4 + 3] = fminf(m[4 * c4 + 3], fmaf(-2.0f, acc[4 * c4 + 3], xi + xj.w));
        }
      }
    }
    if (last_scan) {
#pragma unroll
      for (int size = 2; size <= 32; size <<= 1)
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1)
#pragma unroll
          for (int a = 0; a < 32; ++a) {
            const int p2 = a ^ stride;
            if (p2 > a) {
              const bool up = (a & size) == 0;
              const float lo = fminf(m[a], m[p2]), hi = fmaxf(m[a], m[p2]);
              m[a] = up ? lo : hi;
              m[p2] = up ? hi : lo;
            }
          }
      float tau = -CUDART_INF_F;  // m[k1 - 1] of the ascending array, as a masked maximum (see TcList::kth)
#pragma unroll
      for (int c = 0; c < 32; ++c)
        if (c < k1) tau = fmaxf(tau, m[c]);
      thr = tau + 2.0f * eps;
    }

    // the tile's 256-bit hit mask first, then every lane walks ITS hits (two per step) at its own pace: a warp takes
    // max-over-lanes(hits in the tile) / 2 steps, not the sum over the eight 32-column chunks of the per-chunk maxima
    unsigned hm[kTcTile / 32];
#pragma unroll
    for (int q = 0; q < kTcTile / 32; ++q) hm[q] = 0u;
    if (eval) {  // (uniform over the CTA)
#pragma unroll
    for (int q = 0; q < kTcTile / 32; ++q) {
      float acc[32];
      tc_ld32(trow + (uint32_t)(q * 32), acc);
      const float4 *sx4 = reinterpret_cast<const float4 *>(kTileNorms ? sxx + q * 32 : sxx + t * kTcTile + q * 32);
      unsigned hits = 0u;
#pragma unroll
      for (int c4 = 0; c4 < 8; ++c4) {
        const float4 xj = sx4[c4];
        hits |= (fmaf(-2.0f, acc[4 * c4], xi + xj.x) <= thr ? 1u : 0u) << (4 * c4);
        hits |= (fmaf(-2.0f, acc[4 * c4 + 1], xi + xj.y) <= thr ? 1u : 0u) << (4 * c4 + 1);
        hits |= (fmaf(-2.0f, acc[4 * c4 + 2], xi + xj.z) <= thr ? 1u : 0u) << (4 * c4 + 2);
        hits |= (fmaf(-2.0f, acc[4 * c4 + 3], xi + xj.w) <= thr ? 1u : 0u) << (4 * c4 + 3);
      }
      hm[q] = live ? hits : 0u;
    }
    }
    auto next_hit = [&]() -> int {  // lowest set bit of the 256-bit mask, cleared; -1 when none is left
      unsigned w = 0u;
      int base = -1;
#pragma unroll
      for (int q = kTcTile / 32 - 1; q >= 0; --q)
        if (hm[q]) {
          w = hm[q];
          base = q;
        }
#pragma unroll
      for (int q = 0; q < kTcTile / 32; ++q)
        if (q == base) hm[q] = w & (w - 1u);
      return base < 0 ? -1 : base * 32 + __ffs(w) - 1;
    };
    while (true) {
      const int jr0 = next_hit();
      if (!__any_sync(0xffffffffu, jr0 >= 0)) break;
      if (jr0 >= 0) {
        const int jr1 = next_hit();
        const int jrb = jr1 >= 0 ? jr1 : jr0;
        float d0, d1;
        exact2(jr0, jrb, kTileNorms ? sxx[jr0] : sxx[t * kTcTile + jr0], kTileNorms ? sxx[jrb] : sxx[t * kTcTile + jrb],
               d0, d1);
        if (d0 < top.v[KM - 1]) top.push(d0, t * kTcTile + jr0);
        if (jr1 >= 0 && d1 < top.v[KM - 1]) top.push(d1, t * kTcTile + jr1);
      }
    }
    if (eval) thr = fminf(thr, (k1 == KM ? top.v[KM - 1] : top.kth(k1)) + 2.0f * eps);
    tc_fence_before();
    __syncthreads();  // the accumulator and the B panels are free again
    tc_fence_after();
  }
  if (live) {
    const size_t o = ((size_t)b * K + i) * k1;
#pragma unroll
    for (int s = 0; s < KM; ++s)
      if (s < k1) {
        if (vals) vals[o + s] = top.v[s];
        idx[o + s] = top.id[s];
      }
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

__device__ __forceinline__ void tc_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, "
      "[%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- long lists (33 <= k1 <= 64; DGCNN with k = 40): the same filter and exact evaluation, register budget reworked ----
// A 64-entry (value, index) list takes 128 registers, and knn_tc_fused_kernel<64, 32> already uses 251, so this kernel
// differs from it in three ways (the short-list instantiations stay as they are):
//   * the own row is always re-read from the A panels (as C = 96/128 already do): -C registers at C <= 64;
//   * the threshold sweep and the evaluation sweep are two separate loops, and the list is initialised between them,
//     so the 64 class minima and the 128 list registers are never live together;
//   * the TMEM accumulator is read 16 columns at a time instead of 32.
// The first threshold is the k1-th smallest of 64 column-class minima (class = column mod 64; K >= 256, so tile 0 alone
// already gives every class a real column): k1 <= 64 distinct columns have an approximate distance <= tau, so the
// admission test  approx_j <= (k1-th exact so far) + 2 eps  is the short-list kernel's, and so are values and indices.
template <int C, bool kTileNorms>
__global__ void __launch_bounds__(128, C <= 64 ? 2 : 1)
    knn_tc_long_kernel(const __grid_constant__ CUtensorMap map, int K, int k1, int two_pass,
                       const float *__restrict__ xx, float *__restrict__ vals, int *__restrict__ idx) {
  constexpr int KM = 64;
  constexpr int NP = C / kTcPanelK;
  constexpr int kABytes = kTcRows * 128, kBBytes = kTcTile * 128;
  extern __shared__ __align__(1024) unsigned char smraw[];
  unsigned char *sA = smraw, *sB = smraw + NP * kABytes;
  float *sxx = reinterpret_cast<float *>(sB + NP * kBBytes);
  __shared__ __align__(8) uint64_t bar_a, bar_b, bar_mma;
  __shared__ uint32_t tmem_base_s;
  __shared__ float wmax[4];

  const int b = blockIdx.y, row0 = blockIdx.x * kTcRows;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int ntiles = (K + kTcTile - 1) / kTcTile;

  if (tid == 0) {
    hg_mbar_init(&bar_a, 1);
    hg_mbar_init(&bar_b, 1);
    hg_mbar_init(&bar_mma, 1);
    hg_mbar_init_fence();
  }
  if (warp == 0) {
    __syncwarp();
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(hg_smem_addr(&tmem_base_s))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  float xmax = 0.f;
  if (kTileNorms) {
    for (int j = tid; j < K; j += 128) xmax = fmaxf(xmax, xx[(size_t)b * K + j]);
  } else {
    for (int j = tid; j < ntiles * kTcTile; j += 128) {
      const float v = j < K ? xx[(size_t)b * K + j] : CUDART_INF_F;
      sxx[j] = v;
      if (j < K) xmax = fmaxf(xmax, v);
    }
  }
  xmax = hg_warp_max_f32(xmax);
  if ((tid & 31) == 0) wmax[warp] = xmax;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  xmax = fmaxf(fmaxf(wmax[0], wmax[1]), fmaxf(wmax[2], wmax[3]));

  if (tid == 0) {
    hg_mbar_expect_tx(&bar_a, NP * kABytes);
    for (int p = 0; p < NP; ++p) tc_tma_load_3d(sA + p * kABytes, &map, &bar_a, p * kTcPanelK, row0, b);
  }

  const int i = row0 + tid;
  const bool live = i < K;
  const float xi = live ? (kTileNorms ? xx[(size_t)b * K + i] : sxx[i]) : 0.f;
  const float eps = 1.1f * 0.00390625f * sqrtf(xi * xmax) + 1e-5f * (xi + xmax);
  const uint32_t trow = tmem + ((uint32_t)(warp * 32) << 16);
  const unsigned sw = (unsigned)(tid & 7);
  unsigned phase_b = 0, phase_m = 0;

  // tile t into the B panels, 128 x 256 accumulator into TMEM; every thread waits for both itself
  auto load_mma = [&](int t, bool first) {
    if (tid == 0) {
      hg_mbar_expect_tx(&bar_b, NP * kBBytes);
      for (int p = 0; p < NP; ++p) {
        tc_tma_load_3d(sB + p * kBBytes, &map, &bar_b, p * kTcPanelK, t * kTcTile, b);
        tc_tma_load_3d(sB + p * kBBytes + kABytes, &map, &bar_b, p * kTcPanelK, t * kTcTile + 128, b);
      }
      if (first) tc_mbar_wait(&bar_a, 0);
      tc_mbar_wait(&bar_b, phase_b);
      tc_fence_after();
      constexpr uint32_t idesc = tc_idesc(kTcRows, kTcTile);
#pragma unroll
      for (int p = 0; p < NP; ++p)
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          tc_mma_tf32(tmem, tc_smem_desc(sA + p * kABytes, ks * 32), tc_smem_desc(sB + p * kBBytes, ks * 32), idesc,
                      (p | ks) ? 1u : 0u);
      tc_commit(&bar_mma);
    }
    if (kTileNorms) tc_stage_tile_norms(sxx, xx + (size_t)b * K, K, t, tid);
    if (first) tc_mbar_wait(&bar_a, 0);
    tc_mbar_wait(&bar_b, phase_b);
    phase_b ^= 1;
    tc_mbar_wait(&bar_mma, phase_m);
    phase_m ^= 1;
    __syncwarp();
    tc_fence_after();
    if (kTileNorms) __syncthreads();  // the tile's norms, stored by all four warps
  };
  auto release = [&]() {
    tc_fence_before();
    __syncthreads();  // the accumulator and the B panels are free again
    tc_fence_after();
  };

  // ---- threshold sweep: all tiles (two_pass) or tile 0 only ----
  float thr;
  {
    float m[64];
#pragma unroll
    for (int c = 0; c < 64; ++c) m[c] = CUDART_INF_F;
    const int nscan = two_pass ? ntiles : 1;
    for (int t = 0; t < nscan; ++t) {
      load_mma(t, t == 0);
#pragma unroll 1
      for (int q2 = 0; q2 < kTcTile / 64; ++q2)
#pragma unroll
        for (int h = 0; h < 4; ++h) {  // columns q2 * 64 + h * 16 + c: class h * 16 + c
          float acc[16];
          tc_ld16(trow + (uint32_t)(q2 * 64 + h * 16), acc);
          const float4 *sx4 = reinterpret_cast<const float4 *>((kTileNorms ? sxx : sxx + t * kTcTile) + q2 * 64 + h * 16);
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 xj = sx4[c4];
            float *mm = m + h * 16 + 4 * c4;
            mm[0] = fminf(mm[0], fmaf(-2.0f, acc[4 * c4], xi + xj.x));
            mm[1] = fminf(mm[1], fmaf(-2.0f, acc[4 * c4 + 1], xi + xj.y));
            mm[2] = fminf(mm[2], fmaf(-2.0f, acc[4 * c4 + 2], xi + xj.z));
            mm[3] = fminf(mm[3], fmaf(-2.0f, acc[4 * c4 + 3], xi + xj.w));
          }
        }
      if (two_pass) release();
    }
#pragma unroll
    for (int size = 2; size <= 64; size <<= 1)
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1)
#pragma unroll
        for (int a = 0; a < 64; ++a) {
          const int p2 = a ^ stride;
          if (p2 > a) {
            const bool up = (a & size) == 0;
            const float lo = fminf(m[a], m[p2]), hi = fmaxf(m[a], m[p2]);
            m[a] = up ? lo : hi;
            m[p2] = up ? hi : lo;
          }
        }
    float tau = -CUDART_INF_F;  // m[k1 - 1], as a masked maximum (see TcList::kth)
#pragma unroll
    for (int c = 0; c < 64; ++c)
      if (c < k1) tau = fmaxf(tau, m[c]);
    thr = tau + 2.0f * eps;
  }

  // ---- evaluation sweep (the single-sweep variant evaluates tile 0 from the accumulator it has just scanned) ----
  TcList<KM> top;
  top.init();
  for (int t = 0; t < ntiles; ++t) {
    if (two_pass || t > 0) load_mma(t, false);
    unsigned hm[kTcTile / 32];
#pragma unroll
    for (int q = 0; q < kTcTile / 32; ++q) {
      unsigned hits = 0u;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        float acc[16];
        tc_ld16(trow + (uint32_t)(q * 32 + h * 16), acc);
        const float4 *sx4 = reinterpret_cast<const float4 *>((kTileNorms ? sxx : sxx + t * kTcTile) + q * 32 + h * 16);
#pragma unroll
        for (int c4 = 0; c4 < 4; ++c4) {
          const float4 xj = sx4[c4];
          const int s = h * 16 + 4 * c4;
          hits |= (fmaf(-2.0f, acc[4 * c4], xi + xj.x) <= thr ? 1u : 0u) << s;
          hits |= (fmaf(-2.0f, acc[4 * c4 + 1], xi + xj.y) <= thr ? 1u : 0u) << (s + 1);
          hits |= (fmaf(-2.0f, acc[4 * c4 + 2], xi + xj.z) <= thr ? 1u : 0u) << (s + 2);
          hits |= (fmaf(-2.0f, acc[4 * c4 + 3], xi + xj.w) <= thr ? 1u : 0u) << (s + 3);
        }
      }
      hm[q] = live ? hits : 0u;
    }
    auto next_hit = [&]() -> int {  // lowest set bit of the 256-bit mask, cleared; -1 when none is left
      unsigned w = 0u;
      int base = -1;
#pragma unroll
      for (int q = kTcTile / 32 - 1; q >= 0; --q)
        if (hm[q]) {
          w = hm[q];
          base = q;
        }
#pragma unroll
      for (int q = 0; q < kTcTile / 32; ++q)
        if (q == base) hm[q] = w & (w - 1u);
      return base < 0 ? -1 : base * 32 + __ffs(w) - 1;
    };
    while (true) {
      const int jr0 = next_hit();
      if (!__any_sync(0xffffffffu, jr0 >= 0)) break;
      if (jr0 >= 0) {
        const int jr1 = next_hit();
        const int jrb = jr1 >= 0 ? jr1 : jr0;
        // the reference's sequential FMA chain for columns jr0, jrb (see exact2 in knn_tc_fused_kernel)
        float acc0 = 0.f, acc1 = 0.f;
        const unsigned sw0 = (unsigned)(jr0 & 7), sw1 = (unsigned)(jrb & 7);
#pragma unroll
        for (int p = 0; p < NP; ++p) {
          const unsigned char *r0 = sB + p * kBBytes + jr0 * 128, *r1 = sB + p * kBBytes + jrb * 128;
          const unsigned char *rowi = sA + p * kABytes + tid * 128;
#pragma unroll
          for (int c = 0; c < 8; ++c) {
            const float4 v0 = *reinterpret_cast<const float4 *>(r0 + ((c ^ sw0) << 4));
            const float4 v1 = *reinterpret_cast<const float4 *>(r1 + ((c ^ sw1) << 4));
            const float4 a = *reinterpret_cast<const float4 *>(rowi + ((c ^ sw) << 4));
            acc0 = __fmaf_rn(a.x, v0.x, acc0);
            acc1 = __fmaf_rn(a.x, v1.x, acc1);
            acc0 = __fmaf_rn(a.y, v0.y, acc0);
            acc1 = __fmaf_rn(a.y, v1.y, acc1);
            acc0 = __fmaf_rn(a.z, v0.z, acc0);
            acc1 = __fmaf_rn(a.z, v1.z, acc1);
            acc0 = __fmaf_rn(a.w, v0.w, acc0);
            acc1 = __fmaf_rn(a.w, v1.w, acc1);
          }
        }
        const float *tnorm = kTileNorms ? sxx : sxx + t * kTcTile;
        const float d0 = __fadd_rn(__fadd_rn(__fadd_rn(tnorm[jr0], __fmul_rn(-2.0f, acc0)), xi), 0.0f);
        const float d1 = __fadd_rn(__fadd_rn(__fadd_rn(tnorm[jrb], __fmul_rn(-2.0f, acc1)), xi), 0.0f);
        if (d0 < top.v[KM - 1]) top.push(d0, t * kTcTile + jr0);
        if (jr1 >= 0 && d1 < top.v[KM - 1]) top.push(d1, t * kTcTile + jr1);
      }
    }
    thr = fminf(thr, (k1 == KM ? top.v[KM - 1] : top.kth(k1)) + 2.0f * eps);
    release();
  }
  if (live) {
    const size_t o = ((size_t)b * K + i) * k1;
#pragma unroll
    for (int s = 0; s < KM; ++s)
      if (s < k1) {
        if (vals) vals[o + s] = top.v[s];
        idx[o + s] = top.id[s];
      }
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

template <int C, bool kTileNorms>
int run_tc(const float *pc, const float *xx, int B, int K, int k1, float *vals, int *idx, cudaStream_t stream) {
  EncodeTiledFn enc = encode_tiled();
  HG_REQUIRE(enc != nullptr, HG_E_UNSUPPORTED, "knn (tensor-core path): cuTensorMapEncodeTiled is not available");
  constexpr int NP = C / kTcPanelK;
  const size_t smem = (size_t)NP * (kTcRows + kTcTile) * 128 +
                      (size_t)(kTileNorms ? 1 : (K + kTcTile - 1) / kTcTile) * kTcTile * sizeof(float);
  static HgPerDeviceOnce once;
  if (once.first()) {
    HG_CUDA((cudaFuncSetAttribute(knn_tc_fused_kernel<C, 20, kTileNorms>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)));
    HG_CUDA((cudaFuncSetAttribute(knn_tc_fused_kernel<C, 32, kTileNorms>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)));
    HG_CUDA((cudaFuncSetAttribute(knn_tc_long_kernel<C, kTileNorms>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024)));
  }
  CUtensorMap map;
  const cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)K, (cuuint64_t)B};
  const cuuint64_t gstr[2] = {(cuuint64_t)C * sizeof(float), (cuuint64_t)K * C * sizeof(float)};
  const cuuint32_t box[3] = {kTcPanelK, kTcRows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult cr = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(pc), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  HG_REQUIRE(cr == CUDA_SUCCESS, HG_E_UNSUPPORTED, "knn (tensor-core path): cuTensorMapEncodeTiled failed (%d)", (int)cr);
  dim3 grid((K + kTcRows - 1) / kTcRows, B);
  // threshold from a first, MMA-only sweep over all tiles (default: 130 -> 106 us at 32 x 1024 x 64); hg_tune("knn_tc", 5)
  // forces the single sweep whose threshold starts from tile 0 only
  const int two_pass = g_hg_tune_knn_tc_off == 5 ? 0 : 1;
  if (k1 <= 20)
    knn_tc_fused_kernel<C, 20, kTileNorms><<<grid, 128, smem, stream>>>(map, K, k1, two_pass, xx, vals, idx);
  else if (k1 <= 32)
    knn_tc_fused_kernel<C, 32, kTileNorms><<<grid, 128, smem, stream>>>(map, K, k1, two_pass, xx, vals, idx);
  else
    knn_tc_long_kernel<C, kTileNorms><<<grid, 128, smem, stream>>>(map, K, k1, two_pass, xx, vals, idx);
  HG_CHECK_LAUNCH("knn_tc_fused_kernel");
  return HG_OK;
}

}  // namespace

// Shapes the tensor-core path takes with the cloud's column norms resident: C a multiple of 32 up to 128 (DGCNN: 64, 64,
// 128), clouds of 256..4096 points, lists of up to 64 neighbours.  (The padded 3-D route, hg_knn3.cu, is held to these.)
bool hg_knn_tc_supported(int K, int C, int k1) {
  return (C == 32 || C == 64 || C == 96 || C == 128) && K >= 256 && K <= 4096 && k1 <= 64;
}

// Feature clouds: the same, up to 16384 points (per-tile column norms beyond 4096).
bool hg_knn_tc_supported_feature(int K, int C, int k1) {
  return (C == 32 || C == 64 || C == 96 || C == 128) && K >= 256 && K <= 16384 && k1 <= 64;
}

// xx [B,K] are the reference squared norms (knn_sumsq_kernel).  B <= 65535 (checked by the caller).
int hg_knn_tc_run(const float *pc, const float *xx, int B, int K, int C, int k1, float *vals, int *idx,
                  cudaStream_t stream) {
  const bool tile = K > 4096;
  switch (C) {
    case 32: return tile ? run_tc<32, true>(pc, xx, B, K, k1, vals, idx, stream) : run_tc<32, false>(pc, xx, B, K, k1, vals, idx, stream);
    case 64: return tile ? run_tc<64, true>(pc, xx, B, K, k1, vals, idx, stream) : run_tc<64, false>(pc, xx, B, K, k1, vals, idx, stream);
    case 96: return tile ? run_tc<96, true>(pc, xx, B, K, k1, vals, idx, stream) : run_tc<96, false>(pc, xx, B, K, k1, vals, idx, stream);
    case 128: return tile ? run_tc<128, true>(pc, xx, B, K, k1, vals, idx, stream) : run_tc<128, false>(pc, xx, B, K, k1, vals, idx, stream);
  }
  hg_set_error("knn (tensor-core path): unsupported channel count %d", C);
  return HG_E_UNSUPPORTED;
}
