/*
 * hitgeom.h -- C ABI of libhitgeom.so, the B200-native (sm_100a) replacement for HiT-ADV's point-set
 * geometry hot path.  This is the drop-in boundary: plain pointers and sizes, no torch types.
 *
 * Conventions (all entry points)
 *   - every pointer is a DEVICE pointer to a dense row-major array (the host mirror checks contiguity,
 *     as the reference's CHECK_CONTIGUOUS does, _ext-src/include/utils.h:10-13);
 *   - points are FP32, indices INT32 unless a signature says int64 (torch-level seams);
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and never
 *     synchronises; inputs are borrowed, outputs and workspaces are caller-allocated;
 *   - the return value is 0 on success, a negative HG_E_* code for bad arguments, or a positive
 *     cudaError_t for a launch failure; hg_last_error() returns a thread-local message.  Nothing calls
 *     exit() (the reference does: _ext-src/include/cuda_utils.h:30-39);
 *   - results are deterministic: no floating-point atomics anywhere (the reference's *_grad kernels use
 *     atomicAdd, SURVEY.md section 2.2 K3/K6/K9).
 *
 * Each declaration cites the reference interface it replaces (paths relative to the reference root).
 */
#ifndef HITGEOM_H_
#define HITGEOM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HG_OK 0
#define HG_E_BADARG (-1)      /* null pointer, non-positive size, unsupported k ... */
#define HG_E_WORKSPACE (-2)   /* workspace too small (see the *_workspace_bytes function) */
#define HG_E_UNSUPPORTED (-3) /* shape outside what the kernels implement */

#define HG_MODE_CHAMFER 0
#define HG_MODE_HAUSDORFF 1

typedef void *hgStream; /* cudaStream_t */

int hg_version(void);
const char *hg_last_error(void);
/* SM count, max SM clock [kHz], L2 bytes, global memory bytes of the current device. */
int hg_device_info(int *sm_count, int *clock_khz, long long *l2_bytes, long long *mem_bytes);
/* Measured FP32 FFMA throughput of the current device [TFLOP/s] (independent FFMA chains, no memory traffic): the roofline
 * denominator bench.py reports next to the computed SMs x 128 x 2 x clock figure.  Synchronises the stream. */
int hg_probe_fp32_peak(float *tflops, float *device_scratch, hgStream stream);

/* Every compute entry point below opens an NVTX range named after itself (header-only NVTX v3: free unless nsys / ncu
 * is attached), so a timeline of a reference run shows which reference call each kernel belongs to. */
/* Optional device timing of the hot kernels (used by bench.py for the roofline line).  hg_prof_enable(1) resets
 * the counters and brackets every launch of a tagged kernel with CUDA events on the launching stream;
 * hg_prof_read synchronises those events and returns the summed device time [ms] and the launch count. */
#define HG_PROF_NN_BIDIR 0 /* nn_bidir_d3_kernel  (Chamfer / Hausdorff distance pass) */
#define HG_PROF_KNN 1      /* knn3_kernel         (kNN distance pass + top-k) */
#define HG_PROF_FPS 2      /* fps_kernel */
#define HG_PROF_GROUP 3    /* gather_channel_major_kernel (group_points / gather_points) */
#define HG_PROF_NTAGS 4
/* Development knobs for A/B measurements (not part of the stable ABI; an unknown key returns HG_E_BADARG):
 * "knn_tc" = 1 switches the tensor-core kNN kernel off, 2 forces it for small batches, 5 forces it with the
 * single-sweep threshold;
 * "small_fused" = 1 sends clouds that fit in shared memory down the general finish / kNN-backward kernels as well
 * (same results; the tests run both);
 * "prune" = 0 switches the pruned passes off, "prune_min_n" moves their size threshold, "prune_count" = 1 counts visited
 * leaf pairs, self-kNN drains and orderings; "prune_refit_tol" = rebuild tolerance of an ordering state's refit
 * [permille] (0 = default), "prune_refit_stage" = 1 stages the cloud in shared memory for the refit's gather, 2 reads it
 * from global memory (0 = default). */
int hg_tune(const char *key, int value);
/* Leaf pairs the pruned passes visited and could have visited since the last call: {Chamfer visited, Chamfer total,
 * kNN visited, kNN total}, counted while hg_tune("prune_count", 1) is on.  Synchronises the device. */
int hg_prune_counters(unsigned long long *out4);
/* Drains of the pruned self-kNN search since the last call, counted while hg_tune("prune_count", 1) is on: {leaves
 * drained (per warp of 32 queries), candidates inserted into a query's list, warp rounds of the drains (a round inserts
 * one candidate on every lane that has one left)}.  Synchronises the device. */
int hg_prune_drain_counters(unsigned long long *out3);
/* Ordering builds since the last call, counted per cloud while hg_tune("prune_count", 1) is on: {refit and kept, rebuilt
 * from a state (invalid permutation or degraded leaf boxes), built without a state}.  Synchronises the device. */
int hg_prune_order_counters(unsigned long long *out3);
unsigned long long hg_launch_count(void); /* kernels launched by this library since it was loaded */
void hg_prof_enable(int on);
int hg_prof_read(int tag, float *total_ms, int *launches);
/* Benchmark-only override of the nn_bidir tile shape: T = columns per lane (8 or 16), RB = rows per CTA; 0 = auto. */
void hg_nn_bidir_tune(int T, int RB);
/* Benchmark-only overrides: smallest cloud size whose self-kNN gets grid-seeded thresholds (0 = default), and the
 * seed scan's cell neighbourhood (0 = automatic, 1 = 2x2x2, 2 = 3x3x3). */
void hg_knn_tune(int seed_min_n, int neighbourhood);
/* Test-only override of the streaming 3-D kNN kernel's instantiation: qt = queries per lane (1, 2, 4), gp = candidate
 * pairs per filter bit (2, 4); 0 = chosen from the problem size.  A combination that is not instantiated for the
 * requested k makes the next kNN call fail with HG_E_UNSUPPORTED.  Process-global, not thread-safe. */
void hg_knn_force_shape(int qt, int gp);
/* Benchmark / test-only: largest cloud whose self-kNN takes the small-cloud path (whole cloud resident in shared
 * memory, drain deferred): 0 = default (4096 points), a negative value switches the path off, at most 8192. */
void hg_knn_tune_small(int small_max_n);

/* ---------------------------------------------------------------------------------------------------------
 * util/set_distance.py:15-32,45-48,65-68 -- `_Distance.batch_pairwise_dist` fused with the two `torch.min`
 * reductions; P = (rx_i + ry_j) - 2*zz_ij (FMA-chain dot products) is never materialised.
 *   gts [B,N2,D] ("ori"), preds [B,N1,D] ("adv")
 *   min1/arg1 [B,N1]: for each pred point the nearest gt  (torch.min(P,1)), first index on ties
 *   min2/arg2 [B,N2]: for each gt point the nearest pred (torch.min(P,2)), first index on ties
 * D == 3 runs the register-tiled packed-FP32 kernel; any other D the generic kernel.
 * ------------------------------------------------------------------------------------------------------- */
size_t hg_nn_bidir_workspace_bytes(int B, int N2, int N1, int D);
int hg_nn_bidir_f32(const float *gts, const float *preds, int B, int N2, int N1, int D, float *min1, int *arg1,
                    float *min2, int *arg2, void *workspace, size_t workspace_bytes, hgStream stream);

/* Ordering state for attack loops (CW/kNN.py:77-111 evaluates the losses 2500 times on the same `ori` and on an `adv`
 * that moves by a learning-rate step per iteration).  Clouds of 8192..16384 points take spatially pruned passes that
 * first put every cloud in kd-tree order; a state keeps one cloud batch's permutation (int32 [B,N]) and, per cloud, the
 * quality of the leaf boxes it had when it was built.  A call with a state refits instead of rebuilding: it gathers the
 * points through the stored permutation and recomputes norms and leaf boxes (a pass over memory), and rebuilds, on the
 * device and only for those clouds, the orderings whose permutation is invalid or whose boxes have grown by more than a
 * tolerance.  The state holds nothing specific to a call, so the Chamfer call and the self-kNN call on the same cloud can
 * share one.  Everything read from the state is validated on the device: garbage or stale contents (an uninitialised
 * buffer included) cost speed, never correctness -- results are bit-identical to the stateless calls.  The state is
 * read and written by the call, on its stream: one state must not be used by calls on two streams at the same time.
 * It is ignored and left untouched when the pruned path does not apply (D != 3, N outside the size range,
 * hg_tune("prune", 0)).  The size does not depend on hg_tune, so a caller can allocate once. */
size_t hg_order_state_bytes(int B, int N);
/* hg_nn_bidir_f32 with ordering states for gts [B,N2,3] and preds [B,N1,3]: two distinct buffers, 16-byte aligned;
 * either may be NULL (that cloud is then ordered in the workspace, as hg_nn_bidir_f32 does).  Same workspace. */
int hg_nn_bidir_temporal_f32(const float *gts, const float *preds, int B, int N2, int N1, int D, float *min1, int *arg1,
                             float *min2, int *arg2, void *gts_order, void *preds_order, void *workspace,
                             size_t workspace_bytes, hgStream stream);

/* util/set_distance.py:15-32 `batch_pairwise_dist(x [B,Nx,D], y [B,Ny,D])` -> P [B,Nx,Ny], materialised.
 * Debug / API-completeness entry point: the loss path above never stores P. */
int hg_pairwise_dist_f32(const float *x, const float *y, int B, int Nx, int Ny, int D, float *P, hgStream stream);

/* util/set_distance.py:46-49 (ChamferDistance: torch.mean) and :66-69 (HausdorffDistance: torch.max).
 * loss1/loss2 [B]; hd_arg1/hd_arg2 [B] = first index attaining the max (HAUSDORFF only, may be NULL). */
int hg_set_loss_f32(const float *min1, const float *min2, int B, int N1, int N2, int mode, float *loss1,
                    float *loss2, int *hd_arg1, int *hd_arg2, hgStream stream);

/* Backward of chamfer / hausdorff through the saved indices (what autograd derives for
 * set_distance.py:31,46-49,66-69).  g1/g2 [B] = dL/dloss1, dL/dloss2; either may be NULL = that loss is unused
 * (ChamferDist's default 'adv2ori' never touches loss2): its term and its reverse map are skipped.  grad_preds
 * [B,N1,D] is always written; grad_gts [B,N2,D] may be NULL.  The scatter direction is a deterministic segmented sum. */
size_t hg_set_loss_bwd_workspace_bytes(int B, int N2, int N1);
int hg_set_loss_bwd_f32(const float *gts, const float *preds, const int *arg1, const int *arg2, const int *hd_arg1,
                        const int *hd_arg2, const float *g1, const float *g2, int B, int N2, int N1, int D, int mode,
                        float *grad_preds, float *grad_gts, void *workspace, size_t workspace_bytes, hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * util/dist_utils.py:148-156 (KNNDist) and model/dgcnn_cls.py:8-12 (DGCNN knn): the k1 smallest entries per
 * row of dist[i,j] = (xx_j + (-2*zz_ij)) + xx_i (DGCNN's pairwise_distance is exactly -dist).
 *   pc [B,K,C] point-major; vals [B,K,k1] ascending (may be NULL), idx [B,K,k1], lowest index first on ties.
 *   1 <= k1 <= 64 for every C, k1 <= K (DGCNN's k = 40 on its feature layers included).
 *   C != 3: K <= 12800 for every C; C = 32, 64, 96 or 128 (DGCNN's 64, 64, 128) up to K = 16384, where clouds of more
 *   than 12800 points take the tensor-core kernel only (hg_tune("knn_tc", 1) then fails with HG_E_UNSUPPORTED).
 * ------------------------------------------------------------------------------------------------------- */
size_t hg_knn_self_workspace_bytes(int B, int K, int C, int k1);
int hg_knn_self_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx, void *workspace,
                    size_t workspace_bytes, hgStream stream);

/* The same search inside an attack loop (CW/kNN.py:77-111 calls KNNDist on a slowly moving cloud 2500 times):
 * idx_state [B,K,k1] is caller-owned state.  When state_valid != 0 it holds the neighbour indices an earlier call
 * wrote for a NEARBY cloud of the same shape; re-evaluated at the current coordinates they bound every query's k1-th
 * distance, which replaces the spatial pre-pass (C == 3; ignored otherwise).  The entries are checked (range,
 * distinctness): garbage costs speed, never correctness -- results are identical to hg_knn_self_f32.  On return
 * idx_state holds this call's indices (a copy of idx; idx_state may alias idx). */
int hg_knn_self_temporal_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx, int *idx_state,
                             int state_valid, void *workspace, size_t workspace_bytes, hgStream stream);
/* hg_knn_self_temporal_f32 with an ordering state for pc (see hg_order_state_bytes; NULL = ordered in the workspace):
 * a state the Chamfer call on the same cloud just refit or rebuilt is refit again here.  Same workspace. */
int hg_knn_self_temporal_order_f32(const float *pc, int B, int K, int C, int k1, float *vals, int *idx, int *idx_state,
                                   int state_valid, void *order, void *workspace, size_t workspace_bytes,
                                   hgStream stream);

/* util/dist_utils.py:157-172: value = mean of the k = k1-1 non-first neighbours, threshold mean+alpha*std
 * (unbiased), mask, loss[b] = weights[b] * mean(value*mask).  weights may be NULL (ones). */
int hg_knn_outlier_fwd_f32(const float *vals, int B, int K, int k1, float alpha, const float *weights, float *value,
                           float *mask, float *loss, hgStream stream);
/* backward through the saved indices; g [B] = dL/dloss[b] (weights already folded in by the caller). */
size_t hg_knn_outlier_bwd_workspace_bytes(int B, int K, int k1);
int hg_knn_outlier_bwd_f32(const float *pc, const int *idx, const float *mask, const float *g, int B, int K, int C,
                           int k1, float *grad_pc, void *workspace, size_t workspace_bytes, hgStream stream);

/* pytorch3d.ops.knn_points(p1,p2,K) (requirements.txt:8; call sites ShapeAttack/HiT_ADV.py:78-80,320-321,
 * util/dist_utils.py:482-489, FGM/GeoA3_args.py:284): squared L2 from direct differences, K smallest
 * ascending, int64 indices.  p1 [B,N,3], p2 [B,M,3] -> dists [B,N,K], idx [B,N,K].  K <= 64
 * (HiT_ADV's default curv_loss_knn = 32 asks for 33). */
int hg_knn_points_f32(const float *p1, const float *p2, int B, int N, int M, int K, float *dists, int64_t *idx,
                      hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * model/pointnet2_utils.py torch-level seams (PointNet++ SSG victim, config 3).
 * ------------------------------------------------------------------------------------------------------- */
/* :19-40 square_distance(src [B,N,C], dst [B,M,C]) -> [B,N,M] = ((-2*zz) + rs_n) + rd_m */
int hg_square_distance_f32(const float *src, const float *dst, int B, int N, int M, int C, float *out,
                           hgStream stream);
/* :63-84 farthest_point_sample; start [B] = the torch.randint draw of :75; centroids [B,npoint] int64 */
int hg_fps_torch_f32(const float *xyz, int B, int N, int npoint, const int64_t *start, int64_t *centroids,
                     hgStream stream);
/* :87-107 query_ball_point; radius2 = float32(radius**2); group_idx [B,S,nsample] int64 */
int hg_query_ball_torch_f32(float radius2, int nsample, const float *xyz, const float *new_xyz, int B, int N, int S,
                            int64_t *group_idx, hgStream stream);
/* :43-60 index_points(points [B,N,C], idx [B,M] int64) -> [B,M,C] and its backward (deterministic) */
int hg_index_points_f32(const float *points, const int64_t *idx, int B, int N, int C, int M, float *out,
                        hgStream stream);
size_t hg_index_points_grad_workspace_bytes(int B, int N, int M);
int hg_index_points_grad_f32(const float *grad_out, const int64_t *idx, int B, int N, int C, int M, float *grad_points,
                             void *workspace, size_t workspace_bytes, hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * pointnet2_ops `_ext`: the nine kernel wrappers of pointnet2_ops_lib/pointnet2_ops/_ext-src/src, same
 * argument order as the reference's own C-style seam, plus workspace (grad ops), stream and a return code.
 * ------------------------------------------------------------------------------------------------------- */
/* sampling.cpp:4-6   gather_points_kernel_wrapper       points(b,c,n) idx(b,npoints) -> out(b,c,npoints) */
int hg_p2_gather_points(int b, int c, int n, int npoints, const float *points, const int *idx, float *out,
                        hgStream stream);
/* sampling.cpp:7-9   gather_points_grad_kernel_wrapper  grad_out(b,c,npoints) -> grad_points(b,c,n) */
size_t hg_p2_scatter_workspace_bytes(int b, int n, int nedges);
int hg_p2_gather_points_grad(int b, int c, int n, int npoints, const float *grad_out, const int *idx,
                             float *grad_points, void *workspace, size_t workspace_bytes, hgStream stream);
/* sampling.cpp:11-13 furthest_point_sampling_kernel_wrapper  dataset(b,n,3), temp(b,n) scratch -> idxs(b,m) */
int hg_p2_furthest_point_sampling(int b, int n, int m, const float *dataset, float *temp, int *idxs,
                                  hgStream stream);
/* ball_query.cpp:4-6 query_ball_point_kernel_wrapper  new_xyz(b,m,3) xyz(b,n,3) -> idx(b,m,nsample) */
int hg_p2_ball_query(int b, int n, int m, float radius, int nsample, const float *new_xyz, const float *xyz, int *idx,
                     hgStream stream);
/* group_points.cpp:4-6  group_points_kernel_wrapper  points(b,c,n) idx(b,npoints,nsample) -> out(b,c,npoints,nsample) */
int hg_p2_group_points(int b, int c, int n, int npoints, int nsample, const float *points, const int *idx, float *out,
                       hgStream stream);
/* group_points.cpp:8-10 group_points_grad_kernel_wrapper */
int hg_p2_group_points_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out, const int *idx,
                            float *grad_points, void *workspace, size_t workspace_bytes, hgStream stream);
/* pointnet2_utils.py:279-333 QueryAndGroup.forward after its ball query, fused: out (b, 3+c, npoints, nsample) with
 * rows 0..2 = xyz[idx] - new_xyz and rows 3.. = features[idx] (the reference: two grouping ops, an in-place
 * subtraction and a torch.cat over the full tensor).  xyz (b,n,3), new_xyz (b,npoints,3), features (b,c,n) or NULL
 * with c = 0.  The gradient entry point returns d/d features (b,c,n) and d/d xyz as (b,3,n); either may be NULL;
 * workspace as for group_points_grad (hg_p2_scatter_workspace_bytes(b, n, npoints*nsample)). */
int hg_p2_group_concat(int b, int c, int n, int npoints, int nsample, const float *xyz, const float *new_xyz,
                       const float *features, const int *idx, float *out, hgStream stream);
int hg_p2_group_concat_grad(int b, int c, int n, int npoints, int nsample, const float *grad_out, const int *idx,
                            float *grad_xyz_t, float *grad_features, void *workspace, size_t workspace_bytes,
                            hgStream stream);
/* interpolate.cpp:4-5 three_nn_kernel_wrapper  unknown(b,n,3) known(b,m,3) -> dist2(b,n,3) idx(b,n,3) */
int hg_p2_three_nn(int b, int n, int m, const float *unknown, const float *known, float *dist2, int *idx,
                   hgStream stream);
/* interpolate.cpp:6-8 three_interpolate_kernel_wrapper  points(b,c,m) idx/weight(b,n,3) -> out(b,c,n) */
int hg_p2_three_interpolate(int b, int c, int m, int n, const float *points, const int *idx, const float *weight,
                            float *out, hgStream stream);
/* interpolate.cpp:9-12 three_interpolate_grad_kernel_wrapper  grad_out(b,c,n) -> grad_points(b,c,m) */
int hg_p2_three_interpolate_grad(int b, int c, int n, int m, const float *grad_out, const int *idx,
                                 const float *weight, float *grad_points, void *workspace, size_t workspace_bytes,
                                 hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * "Next" row 8f#1: the fused HiT-ADV deformation, ShapeAttack/HiT_ADV.py:168-175 + kernel_density :298-304.
 *   ori [B,3,K], centers [B,3,J] (channel-first, as the attack holds them), perturb [B,J,3], delta [B,J]
 *   out [B,3,K] = sum_j (x + p_j) w_j / sum_j w_j,  w_j = exp(-||x - c_j|| / (2 delta_j^2));  deno [B,K] = sum_j w_j
 * The backward returns the gradients w.r.t. the two optimised tensors (ori / centers are constants in the attack).
 * ------------------------------------------------------------------------------------------------------- */
int hg_hitadv_deform_fwd_f32(const float *ori, const float *centers, const float *perturb, const float *delta, int B,
                             int K, int J, float *out, float *deno, hgStream stream);
int hg_hitadv_deform_bwd_f32(const float *ori, const float *centers, const float *perturb, const float *delta,
                             const float *out, const float *deno, const float *grad_out, int B, int K, int J,
                             float *grad_perturb, float *grad_delta, hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * Row a9' / "next" row 8f#3: DGCNN edge features, model/dgcnn_cls.py:16-43 get_graph_feature (after its kNN).
 *   x [B,C,N] channel-first features, idx [B,N,k] int64 neighbour indices (as torch.topk / model_seams.knn give them)
 *   out [B,2C,N,k]:  out[b,c,n,t] = x[b,c,idx[b,n,t]] - x[b,c,n],   out[b,C+c,n,t] = x[b,c,n]
 * written once in its final layout (the reference goes through gather + repeat + cat + permute().contiguous()).
 * The backward sums the incoming edges through a CSR reverse map in ascending edge order (deterministic; the
 * reference's index_put_(accumulate=True) uses floating-point atomics).  Any N with N*k < 2^31, both directions.
 * ------------------------------------------------------------------------------------------------------- */
int hg_edge_feature_f32(const float *x, const int64_t *idx, int B, int C, int N, int k, float *out, hgStream stream);
size_t hg_edge_feature_grad_workspace_bytes(int B, int N, int k);
int hg_edge_feature_grad_f32(const float *grad_out, const int64_t *idx, int B, int C, int N, int k, float *grad_x,
                             void *workspace, size_t workspace_bytes, hgStream stream);

/* ---------------------------------------------------------------------------------------------------------
 * End-to-end entry point on HOST buffers: one CW-kNN distance step (CW/kNN.py:104-108 calling
 * util/dist_utils.py:258-294 ChamferkNNDist(chamfer_method, knn_k, knn_alpha, chamfer_weight, knn_weight) with
 * batch_avg=True) -- the exception to "every pointer is a device pointer": adv_h, ori_h [B,N,3], weights_h [B] or NULL,
 * cloud_loss_h [B], grad_adv_h [B,N,3] and loss_h [1] are HOST pointers (page-locked memory lets the copies overlap).
 *   cloud_loss[b] = w_b (chamfer_weight * chamfer_b + knn_weight * knn_b);  loss = mean_b cloud_loss[b];
 *   grad_adv = d loss / d adv.   chamfer_method: 0 'adv2ori', 1 'ori2adv', 2 'both' (dist_utils.py:44-80).
 * The batch is pipelined in chunks of `chunk_clouds` over two streams with their own device buffers (owned by the
 * session), so host<->device copies hide behind the kernels; the call returns when loss and gradient are in place.
 * A session serves any B and any knn_k <= knn_k_max for its N; it lives on the device current at creation (calls
 * switch to that device and restore the caller's) and is not thread-safe.
 * ------------------------------------------------------------------------------------------------------- */
typedef struct hgHostStep hgHostStep;
hgHostStep *hg_host_step_create(int N, int chunk_clouds, int knn_k_max); /* NULL on failure (hg_last_error) */
void hg_host_step_destroy(hgHostStep *session);
int hg_chamfer_knn_step_host_f32(hgHostStep *session, const float *adv_h, const float *ori_h, int B, int chamfer_method,
                                 int knn_k, float knn_alpha, float chamfer_weight, float knn_weight,
                                 const float *weights_h, float *loss_h, float *cloud_loss_h, float *grad_adv_h);

#ifdef __cplusplus
}
#endif
#endif /* HITGEOM_H_ */
