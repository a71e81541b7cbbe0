"""Tensor-level entry points: thin wrappers that hand raw device pointers to the C ABI (include/hitgeom.h)
and the `torch.autograd.Function`s whose backward reuses the saved nearest-neighbour indices.

No arithmetic on point data happens in Python/PyTorch here; torch only allocates outputs and workspaces."""
import ctypes

import torch

from . import _lib
from ._lib import HitgeomError, check, lib, ptr, require, stream_ptr, workspace

MODE_CHAMFER, MODE_HAUSDORFF = 0, 1


def _on_tensor_device(fn):
    """Run `fn` with the CUDA device of its first CUDA-tensor argument current (and the caller's restored): the C ABI
    launches on `torch.cuda.current_stream()`, which belongs to the CURRENT device -- the reference's bindings have no
    device guard either (SURVEY.md section 8b), here a tensor on another GPU must not launch on the wrong one."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kw):
        for a in args:
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if a.device.index != torch.cuda.current_device():
                    with torch.cuda.device(a.device):
                        return fn(*args, **kw)
                break
        return fn(*args, **kw)

    return wrapper


# ------------------------------------------------------------------------------------------------------------
# set distance (util/set_distance.py)
# ------------------------------------------------------------------------------------------------------------
def order_state(B, N, device):
    """A kd-tree ordering state for a batch of B clouds of N points (hg_order_state_bytes): uint8, zero-filled, so the
    first call that uses it builds.  Hand it to `nn_bidir` / `knn_self` for the same cloud on later calls, which then
    refit the stored ordering instead of rebuilding it; the results do not depend on its contents."""
    return torch.zeros(max(int(lib().hg_order_state_bytes(int(B), int(N))), 16), dtype=torch.uint8, device=device)


def _check_order(order, B, N, dev, name):
    if order is None:
        return
    require(order, name, dtype=torch.uint8)
    if order.device != dev or order.numel() < lib().hg_order_state_bytes(B, N):
        raise RuntimeError(f"{name} must be an order_state({B}, {N}) tensor on {dev}")


@_on_tensor_device
def nn_bidir(gts, preds, gts_order=None, preds_order=None):
    """Fused `batch_pairwise_dist(gts, preds)` + `torch.min(P,1)` + `torch.min(P,2)` (set_distance.py:15-48).

    gts [B,N2,D], preds [B,N1,D] -> (min1 [B,N1], arg1 [B,N1] int32, min2 [B,N2], arg2 [B,N2] int32).
    `gts_order` / `preds_order` (optional, `order_state(B, N2 | N1, device)`): ordering states of the two clouds
    (hg_nn_bidir_temporal_f32); the results do not depend on them."""
    require(gts, "gts", ndim=3)
    require(preds, "preds", ndim=3)
    B, N2, D = gts.shape
    if preds.shape[0] != B or preds.shape[2] != D:
        raise RuntimeError(f"shape mismatch: gts {tuple(gts.shape)} vs preds {tuple(preds.shape)}")
    N1 = preds.shape[1]
    dev = gts.device
    min1 = torch.empty((B, N1), dtype=torch.float32, device=dev)
    min2 = torch.empty((B, N2), dtype=torch.float32, device=dev)
    arg1 = torch.empty((B, N1), dtype=torch.int32, device=dev)
    arg2 = torch.empty((B, N2), dtype=torch.int32, device=dev)
    nbytes = lib().hg_nn_bidir_workspace_bytes(B, N2, N1, D)
    ws = workspace(nbytes, dev)
    if gts_order is None and preds_order is None:
        check(lib().hg_nn_bidir_f32(ptr(gts), ptr(preds), B, N2, N1, D, ptr(min1), ptr(arg1), ptr(min2), ptr(arg2),
                                    ptr(ws), ws.numel(), stream_ptr()), "hg_nn_bidir_f32")
        return min1, arg1, min2, arg2
    _check_order(gts_order, B, N2, dev, "gts_order")
    _check_order(preds_order, B, N1, dev, "preds_order")
    check(lib().hg_nn_bidir_temporal_f32(ptr(gts), ptr(preds), B, N2, N1, D, ptr(min1), ptr(arg1), ptr(min2), ptr(arg2),
                                         ptr(gts_order), ptr(preds_order), ptr(ws), ws.numel(), stream_ptr()),
          "hg_nn_bidir_temporal_f32")
    return min1, arg1, min2, arg2


@_on_tensor_device
def pairwise_dist(x, y):
    require(x, "x", ndim=3)
    require(y, "y", ndim=3)
    B, Nx, D = x.shape
    Ny = y.shape[1]
    P = torch.empty((B, Nx, Ny), dtype=torch.float32, device=x.device)
    check(lib().hg_pairwise_dist_f32(ptr(x), ptr(y), B, Nx, Ny, D, ptr(P), stream_ptr()), "hg_pairwise_dist_f32")
    return P


@_on_tensor_device
def set_loss(min1, min2, mode):
    B, N1 = min1.shape
    N2 = min2.shape[1]
    dev = min1.device
    loss1 = torch.empty(B, dtype=torch.float32, device=dev)
    loss2 = torch.empty(B, dtype=torch.float32, device=dev)
    hd1 = torch.empty(B, dtype=torch.int32, device=dev) if mode == MODE_HAUSDORFF else None
    hd2 = torch.empty(B, dtype=torch.int32, device=dev) if mode == MODE_HAUSDORFF else None
    check(lib().hg_set_loss_f32(ptr(min1), ptr(min2), B, N1, N2, mode, ptr(loss1), ptr(loss2), ptr(hd1), ptr(hd2),
                                stream_ptr()), "hg_set_loss_f32")
    return loss1, loss2, hd1, hd2


@_on_tensor_device
def set_loss_bwd(gts, preds, arg1, arg2, hd1, hd2, g1, g2, mode, want_gts):
    B, N2, D = gts.shape
    N1 = preds.shape[1]
    dev = gts.device
    grad_preds = torch.empty_like(preds)
    grad_gts = torch.empty_like(gts) if want_gts else None
    ws = workspace(lib().hg_set_loss_bwd_workspace_bytes(B, N2, N1), dev)
    check(lib().hg_set_loss_bwd_f32(ptr(gts), ptr(preds), ptr(arg1), ptr(arg2), ptr(hd1), ptr(hd2), ptr(g1), ptr(g2), B,
                                    N2, N1, D, mode, ptr(grad_preds), ptr(grad_gts), ptr(ws), ws.numel(),
                                    stream_ptr()), "hg_set_loss_bwd_f32")
    return grad_preds, grad_gts


class shared_distance_pass:
    """`with shared_distance_pass(): loss = chamfer(adv, ori) + hausdorff(adv, ori)` -- inside the block, Chamfer and
    Hausdorff losses of the SAME pair of tensors share one distance pass (the reference builds P twice,
    set_distance.py:44,61; SURVEY.md 8d counts one).  Sharing is keyed on tensor identity + version and is only active
    inside the block: the caller asserts that the clouds are not modified through `.data` between the two calls."""
    _depth = 0
    _entries = []

    def __enter__(self):
        shared_distance_pass._depth += 1
        return self

    def __exit__(self, *exc):
        shared_distance_pass._depth -= 1
        if shared_distance_pass._depth == 0:
            shared_distance_pass._entries.clear()
        return False

    @staticmethod
    def lookup(preds, gts, preds_c, gts_c, preds_order=None, gts_order=None):
        if shared_distance_pass._depth == 0:
            return nn_bidir(gts_c, preds_c, gts_order, preds_order)
        key = (preds_c.data_ptr(), preds._version, gts_c.data_ptr(), gts._version, tuple(preds_c.shape),
               tuple(gts_c.shape), stream_ptr())
        for k, _, res in shared_distance_pass._entries:
            if k == key:
                return res
        res = nn_bidir(gts_c, preds_c, gts_order, preds_order)
        # the entry keeps its inputs alive, so their addresses cannot be recycled for other tensors meanwhile
        shared_distance_pass._entries.append((key, (preds, gts, preds_c, gts_c), res))
        return res


class SetDistanceFn(torch.autograd.Function):
    """(preds, gts) -> (loss1 [B], loss2 [B]) for Chamfer (mode 0) / Hausdorff (mode 1); optional ordering states of
    the two clouds (`order_state`)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, preds, gts, mode, preds_order=None, gts_order=None):
        preds_c = preds.detach().contiguous()
        gts_c = gts.detach().contiguous()
        min1, arg1, min2, arg2 = shared_distance_pass.lookup(preds, gts, preds_c, gts_c, preds_order, gts_order)
        loss1, loss2, hd1, hd2 = set_loss(min1, min2, mode)
        ctx.mode = mode
        # save_for_backward (not a plain attribute): preds_c / gts_c alias the caller's storage when it is contiguous,
        # and an in-place update between forward and backward must raise, as it does for the reference's autograd graph
        ctx.save_for_backward(preds, gts, arg1, arg2, hd1, hd2)
        ctx.set_materialize_grads(False)  # an unused loss arrives as None, and its backward work is skipped
        return loss1, loss2

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g1, g2):
        preds, gts, arg1, arg2, hd1, hd2 = ctx.saved_tensors
        preds_c, gts_c = preds.detach().contiguous(), gts.detach().contiguous()
        B = preds_c.shape[0]
        dev = preds_c.device
        need_p, need_g = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if g1 is None and g2 is None:
            return ((torch.zeros_like(preds_c) if need_p else None), (torch.zeros_like(gts_c) if need_g else None), None,
                    None, None)
        g1 = None if g1 is None else g1.to(torch.float32).contiguous()
        g2 = None if g2 is None else g2.to(torch.float32).contiguous()
        grad_preds, grad_gts = set_loss_bwd(gts_c, preds_c, arg1, arg2, hd1, hd2, g1, g2, ctx.mode, need_g)
        return (grad_preds if need_p else None), (grad_gts if need_g else None), None, None, None


def _as_points(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (hitgeom has no CPU path)")
    if t.dtype != torch.float32:
        raise RuntimeError(f"{name} must be float32, got {t.dtype}")
    if t.dim() != 3:
        raise RuntimeError(f"{name} must be [B,N,D], got shape {tuple(t.shape)}")
    return t


def chamfer_losses(preds, gts, preds_order=None, gts_order=None):
    """`ChamferDistance.forward(preds, gts)` (set_distance.py:40-50) -> (loss1 [B], loss2 [B])."""
    return SetDistanceFn.apply(_as_points(preds, "preds"), _as_points(gts, "gts"), MODE_CHAMFER, preds_order, gts_order)


def hausdorff_losses(preds, gts, preds_order=None, gts_order=None):
    """`HausdorffDistance.forward(preds, gts)` (set_distance.py:58-70)."""
    return SetDistanceFn.apply(_as_points(preds, "preds"), _as_points(gts, "gts"), MODE_HAUSDORFF, preds_order,
                               gts_order)


# ------------------------------------------------------------------------------------------------------------
# kNN (util/dist_utils.py KNNDist, model/dgcnn_cls.py knn, pytorch3d.ops.knn_points)
# ------------------------------------------------------------------------------------------------------------
@_on_tensor_device
def knn_self(pc, k1, want_vals=True, state=None, state_valid=False, order=None):
    """k1 smallest per row of dist[i,j] = (xx_j + (-2 zz_ij)) + xx_i.  pc [B,K,C] point-major.

    1 <= k1 <= min(64, K) for every C.  Returns (vals [B,K,k1] ascending or None, idx [B,K,k1] int32).  `state` (optional int32 [B,K,k1], caller-owned):
    the indices of an earlier call on a nearby cloud, used as temporal seeds when `state_valid`, and overwritten with
    this call's indices (hg_knn_self_temporal_f32); `order` (optional, `order_state(B, K, device)`): the cloud's
    ordering state (hg_knn_self_temporal_order_f32).  The results depend on neither."""
    require(pc, "pc", ndim=3)
    B, K, C = pc.shape
    dev = pc.device
    vals = torch.empty((B, K, k1), dtype=torch.float32, device=dev) if want_vals else None
    idx = torch.empty((B, K, k1), dtype=torch.int32, device=dev)
    ws = workspace(lib().hg_knn_self_workspace_bytes(B, K, C, k1), dev)
    if state is not None:
        require(state, "state", dtype=torch.int32, ndim=3)
        if tuple(state.shape) != (B, K, k1) or state.device != dev:
            raise RuntimeError(f"state must be an int32 [{B},{K},{k1}] tensor on {dev}")
    if order is None:
        check(lib().hg_knn_self_temporal_f32(ptr(pc), B, K, C, k1, ptr(vals), ptr(idx), ptr(state),
                                             1 if state_valid else 0, ptr(ws), ws.numel(), stream_ptr()),
              "hg_knn_self_temporal_f32")
        return vals, idx
    _check_order(order, B, K, dev, "order")
    check(lib().hg_knn_self_temporal_order_f32(ptr(pc), B, K, C, k1, ptr(vals), ptr(idx), ptr(state),
                                               1 if state_valid else 0, ptr(order), ptr(ws), ws.numel(), stream_ptr()),
          "hg_knn_self_temporal_order_f32")
    return vals, idx


class KnnOutlierFn(torch.autograd.Function):
    """pc [B,K,3] point-major -> per-sample kNN-outlier loss [B] (dist_utils.py:148-167, unit weights)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, pc, k, alpha, state=None, state_valid=False, order=None):
        pc_c = pc.detach().contiguous()
        B, K, C = pc_c.shape
        dev = pc_c.device
        vals, idx = knn_self(pc_c, k + 1, state=state, state_valid=state_valid, order=order)
        value = torch.empty((B, K), dtype=torch.float32, device=dev)
        mask = torch.empty((B, K), dtype=torch.float32, device=dev)
        loss = torch.empty(B, dtype=torch.float32, device=dev)
        check(lib().hg_knn_outlier_fwd_f32(ptr(vals), B, K, k + 1, float(alpha), None, ptr(value), ptr(mask), ptr(loss),
                                           stream_ptr()), "hg_knn_outlier_fwd_f32")
        ctx.save_for_backward(pc, idx, mask)
        ctx.k1 = k + 1
        return loss

    @staticmethod
    @_on_tensor_device
    def backward(ctx, g):
        pc, idx, mask = ctx.saved_tensors
        pc_c = pc.detach().contiguous()
        B, K, C = pc_c.shape
        g = g.to(torch.float32).contiguous()
        grad = torch.empty_like(pc_c)
        ws = workspace(lib().hg_knn_outlier_bwd_workspace_bytes(B, K, ctx.k1), pc_c.device)
        check(lib().hg_knn_outlier_bwd_f32(ptr(pc_c), ptr(idx), ptr(mask), ptr(g), B, K, C, ctx.k1, ptr(grad), ptr(ws),
                                           ws.numel(), stream_ptr()), "hg_knn_outlier_bwd_f32")
        return grad, None, None, None, None, None


def knn_outlier_loss(pc, k, alpha, state=None, state_valid=False, order=None):
    return KnnOutlierFn.apply(_as_points(pc, "pc"), int(k), float(alpha), state, bool(state_valid), order)


@_on_tensor_device
def knn_points_raw(p1, p2, K):
    require(p1, "p1", ndim=3)
    require(p2, "p2", ndim=3)
    B, N, _ = p1.shape
    M = p2.shape[1]
    dists = torch.empty((B, N, K), dtype=torch.float32, device=p1.device)
    idx = torch.empty((B, N, K), dtype=torch.int64, device=p1.device)
    check(lib().hg_knn_points_f32(ptr(p1), ptr(p2), B, N, M, K, ptr(dists), ptr(idx), stream_ptr()), "hg_knn_points_f32")
    return dists, idx


# ------------------------------------------------------------------------------------------------------------
# torch-level seams of model/pointnet2_utils.py
# ------------------------------------------------------------------------------------------------------------
@_on_tensor_device
def square_distance(src, dst):
    require(src, "src", ndim=3)
    require(dst, "dst", ndim=3)
    B, N, C = src.shape
    M = dst.shape[1]
    out = torch.empty((B, N, M), dtype=torch.float32, device=src.device)
    check(lib().hg_square_distance_f32(ptr(src), ptr(dst), B, N, M, C, ptr(out), stream_ptr()), "hg_square_distance_f32")
    return out


@_on_tensor_device
def fps_torch(xyz, npoint, start):
    require(xyz, "xyz", ndim=3)
    require(start, "start", dtype=torch.int64, ndim=1)
    B, N, _ = xyz.shape
    out = torch.empty((B, npoint), dtype=torch.int64, device=xyz.device)
    check(lib().hg_fps_torch_f32(ptr(xyz), B, N, npoint, ptr(start), ptr(out), stream_ptr()), "hg_fps_torch_f32")
    return out


@_on_tensor_device
def query_ball_torch(radius, nsample, xyz, new_xyz):
    require(xyz, "xyz", ndim=3)
    require(new_xyz, "new_xyz", ndim=3)
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    out = torch.empty((B, S, nsample), dtype=torch.int64, device=xyz.device)
    r2 = float(torch.tensor(radius ** 2, dtype=torch.float32))  # the float32 rounding torch applies to the scalar
    check(lib().hg_query_ball_torch_f32(r2, nsample, ptr(xyz), ptr(new_xyz), B, N, S, ptr(out), stream_ptr()),
          "hg_query_ball_torch_f32")
    return out


class IndexPointsFn(torch.autograd.Function):
    """points [B,N,C], idx [B,M] int64 -> [B,M,C]; backward is a deterministic segmented sum."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, points, idx):
        pts = points.detach().contiguous()
        require(pts, "points", ndim=3)
        require(idx, "idx", dtype=torch.int64, ndim=2)
        if idx.device != pts.device or idx.shape[0] != pts.shape[0]:
            raise RuntimeError(f"index_points: idx {tuple(idx.shape)} on {idx.device} does not match points "
                               f"{tuple(pts.shape)} on {pts.device}")
        B, N, C = pts.shape
        M = idx.shape[1]
        out = torch.empty((B, M, C), dtype=torch.float32, device=pts.device)
        check(lib().hg_index_points_f32(ptr(pts), ptr(idx), B, N, C, M, ptr(out), stream_ptr()), "hg_index_points_f32")
        ctx.save_for_backward(idx)
        ctx.n_points = N
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, grad_out):
        (idx,), N = ctx.saved_tensors, ctx.n_points
        g = grad_out.to(torch.float32).contiguous()
        B, M, C = g.shape
        grad = torch.empty((B, N, C), dtype=torch.float32, device=g.device)
        ws = workspace(lib().hg_index_points_grad_workspace_bytes(B, N, M), g.device)
        check(lib().hg_index_points_grad_f32(ptr(g), ptr(idx), B, N, C, M, ptr(grad), ptr(ws), ws.numel(), stream_ptr()),
              "hg_index_points_grad_f32")
        return grad, None


class DeformFn(torch.autograd.Function):
    """Fused HiT-ADV deformation (HiT_ADV.py:168-175,298-304): (ori [B,3,K], centers [B,3,J], perturb [B,J,3],
    delta [B,J]) -> deformed cloud [B,3,K]; differentiable in perturb and delta."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, ori, centers, perturb, delta):
        ori_c, cen_c = ori.detach().contiguous(), centers.detach().contiguous()
        per_c, del_c = perturb.detach().contiguous(), delta.detach().contiguous()
        for t, name in ((ori_c, "ori"), (cen_c, "centers"), (per_c, "perturb"), (del_c, "delta")):
            require(t, name)
        B, _, K = ori_c.shape
        J = cen_c.shape[2]
        out = torch.empty_like(ori_c)
        deno = torch.empty((B, K), dtype=torch.float32, device=ori_c.device)
        check(lib().hg_hitadv_deform_fwd_f32(ptr(ori_c), ptr(cen_c), ptr(per_c), ptr(del_c), B, K, J, ptr(out), ptr(deno),
                                             stream_ptr()), "hg_hitadv_deform_fwd_f32")
        ctx.save_for_backward(ori, centers, perturb, delta, out, deno)
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, grad_out):
        ori, centers, perturb, delta, out, deno = ctx.saved_tensors
        ori_c, cen_c = ori.detach().contiguous(), centers.detach().contiguous()
        per_c, del_c = perturb.detach().contiguous(), delta.detach().contiguous()
        B, _, K = ori_c.shape
        J = cen_c.shape[2]
        g = grad_out.to(torch.float32).contiguous()
        gp = torch.empty_like(per_c)
        gd = torch.empty_like(del_c)
        check(lib().hg_hitadv_deform_bwd_f32(ptr(ori_c), ptr(cen_c), ptr(per_c), ptr(del_c), ptr(out), ptr(deno), ptr(g),
                                             B, K, J, ptr(gp), ptr(gd), stream_ptr()), "hg_hitadv_deform_bwd_f32")
        return None, None, gp, gd


def hitadv_deform(ori, centers, perturb, delta):
    return DeformFn.apply(ori, centers, perturb, delta)


class EdgeFeatureFn(torch.autograd.Function):
    """DGCNN edge features (dgcnn_cls.py:16-43): x [B,C,N], idx [B,N,k] int64 -> [B,2C,N,k] = cat(x_nbr - x, x)."""

    @staticmethod
    @_on_tensor_device
    def forward(ctx, x, idx):
        xc = x.detach().contiguous()
        require(xc, "x")
        ic = idx.contiguous()
        if ic.dtype != torch.int64 or not ic.is_cuda:
            raise HitgeomError("edge_feature: idx must be a CUDA int64 tensor [B,N,k]")
        B, C, N = xc.shape
        k = ic.shape[2]
        out = torch.empty((B, 2 * C, N, k), dtype=torch.float32, device=xc.device)
        check(lib().hg_edge_feature_f32(ptr(xc), ptr(ic), B, C, N, k, ptr(out), stream_ptr()), "hg_edge_feature_f32")
        ctx.save_for_backward(ic)
        ctx.channels = C
        return out

    @staticmethod
    @_on_tensor_device
    def backward(ctx, grad_out):
        (idx,), C = ctx.saved_tensors, ctx.channels
        g = grad_out.to(torch.float32).contiguous()
        B, _, N, k = g.shape
        grad = torch.empty((B, C, N), dtype=torch.float32, device=g.device)
        ws = workspace(lib().hg_edge_feature_grad_workspace_bytes(B, N, k), g.device)
        check(lib().hg_edge_feature_grad_f32(ptr(g), ptr(idx), B, C, N, k, ptr(grad), ptr(ws), ws.numel(), stream_ptr()),
              "hg_edge_feature_grad_f32")
        return grad, None


def edge_feature(x, idx):
    return EdgeFeatureFn.apply(x, idx)


def tune_nn_bidir(T=0, RB=0):
    """Benchmark-only override of the nn_bidir tile shape (0 = automatic)."""
    lib().hg_nn_bidir_tune(int(T), int(RB))


def force_knn_shape(qt=0, gp=0):
    """Test-only override of the streaming kNN kernel's instantiation (queries per lane, pairs per filter bit)."""
    lib().hg_knn_force_shape(int(qt), int(gp))


def prune_order_counters():
    """Ordering builds of the pruned path since the last call, per cloud, while hg_tune("prune_count", 1) is on:
    (refit and kept, rebuilt from a state, built without a state).  Synchronises the device."""
    out = (ctypes.c_ulonglong * 3)()
    check(lib().hg_prune_order_counters(out), "hg_prune_order_counters")
    return tuple(int(v) for v in out)


def tune_knn_small(small_max_n=0):
    """Benchmark / test-only: largest cloud on the small-cloud kNN path (0 = default, negative = off)."""
    lib().hg_knn_tune_small(int(small_max_n))


__all__ = [n for n in dir() if not n.startswith("_")]
_ = _lib
