"""Drop-in mirror of the hot-path loss classes of the reference's `util/dist_utils.py`:
`ChamferDist` (:44-80), `HausdorffDist` (:83-119), `KNNDist` (:122-175), `ChamferkNNDist` (:258-294) and
`L2Dist` (:15-41, trivial, kept so that `from util.dist_utils import *` users find it).

Same constructor arguments, same `forward(adv_pc, ori_pc, weights=None, batch_avg=True)` contract, same
return values (0-d tensor, or [B] with `batch_avg=False`); weights may arrive as float64 CPU tensors
(CW/Perturb.py:148-150) and are moved with `.float().cuda()` exactly as the reference does.
"""
import torch
import torch.nn as nn

from . import functional as F
from .functional import shared_distance_pass  # noqa: F401  (opt-in: Chamfer + Hausdorff of one pair share a pass)
from .set_distance import chamfer, hausdorff


def _weights(weights, B, device):
    """`weights.float().cuda()` of the reference (dist_utils.py:76); None means unit weights, for which the
    multiplication is skipped (x * 1.0 == x exactly) instead of building a ones tensor on the host every call."""
    if weights is None:
        return None
    return weights.float().to(device)


def _finish(loss, weights, batch_avg):
    if weights is not None:
        loss = loss * weights
    if batch_avg:
        return loss.mean()
    return loss


class L2Dist(nn.Module):
    def __init__(self):
        super(L2Dist, self).__init__()

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        B = adv_pc.shape[0]
        weights = _weights(weights, B, adv_pc.device)
        dist = torch.sqrt(torch.sum((adv_pc - ori_pc) ** 2, dim=[1, 2]) + torch.tensor(1e-7))
        return _finish(dist, weights, batch_avg)


def _order(store, role, t):
    """The ordering state of cloud `t` [B,N,3] in role 'ori' / 'adv' (one per shape and device), allocated on first use
    (zero-filled: the first call builds).  None where the ordering does not apply (not a 3-D CUDA cloud)."""
    if not (t.is_cuda and t.dim() == 3 and t.shape[2] == 3):
        return None
    key = (role, tuple(t.shape), t.device)
    s = store.get(key)
    if s is None:
        s = store[key] = F.order_state(t.shape[0], t.shape[1], t.device)
    return s


class _TemporalOrders:
    """`temporal_seeds(True)` for the set distances (an addition): keep the kd-tree ordering of `adv` and `ori` between
    calls, so that clouds of 8192..16384 points refit the previous call's ordering instead of rebuilding it
    (hg_nn_bidir_temporal_f32).  Meant for attack loops, where `ori` stays put and `adv` moves by a learning-rate step
    per call; the loss and its gradient are the same bits either way.  The states are per (role, batch shape, device) and
    belong to this module: a module must not run on two streams at once.  [B,3,K] inputs (HiT-ADV's channel-first call)
    are not 3-D point clouds and take no state."""

    def temporal_seeds(self, on=True):
        self.temporal = bool(on)
        self._orders = {}
        return self

    def _losses(self, fn, adv_pc, ori_pc):
        po, go = _order(self._orders, "adv", adv_pc), _order(self._orders, "ori", ori_pc)
        if po is not None and go is not None:
            return fn(adv_pc, ori_pc, po, go)
        return fn(adv_pc, ori_pc)


def _select(loss1, loss2, method):
    if method == 'adv2ori':
        return loss1
    elif method == 'ori2adv':
        return loss2
    return (loss1 + loss2) / 2.


class ChamferDist(_TemporalOrders, nn.Module):
    """Same constructor as the reference; `temporal_seeds(True)`: see _TemporalOrders."""

    def __init__(self, method='adv2ori'):
        super(ChamferDist, self).__init__()
        self.method = method

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        B = adv_pc.shape[0]
        # (getattr: install.patch_reference() binds this forward to the REFERENCE's class, which has no temporal state)
        if getattr(self, "temporal", False):
            loss1, loss2 = self._losses(F.chamfer_losses, adv_pc, ori_pc)
        else:
            loss1, loss2 = chamfer(adv_pc, ori_pc)  # [B], adv2ori, ori2adv
        loss = _select(loss1, loss2, self.method)
        return _finish(loss, _weights(weights, B, loss.device), batch_avg)


class HausdorffDist(_TemporalOrders, nn.Module):
    """Same constructor as the reference; `temporal_seeds(True)`: see _TemporalOrders."""

    def __init__(self, method='adv2ori'):
        super(HausdorffDist, self).__init__()
        self.method = method

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        B = adv_pc.shape[0]
        # (getattr: install.patch_reference() binds this forward to the REFERENCE's class, which has no temporal state)
        if getattr(self, "temporal", False):
            loss1, loss2 = self._losses(F.hausdorff_losses, adv_pc, ori_pc)
        else:
            loss1, loss2 = hausdorff(adv_pc, ori_pc)
        loss = _select(loss1, loss2, self.method)
        return _finish(loss, _weights(weights, B, loss.device), batch_avg)


class KNNDist(nn.Module):
    """Same constructor as the reference.  `temporal_seeds(True)` (an addition) keeps the neighbour indices of the
    previous call as state and hands them to the next call as seeds: inside an attack loop (CW/kNN.py:77-111) the cloud
    moves by a learning-rate step per iteration, so they bound every k-th distance almost tightly and replace the
    spatial pre-pass.  Clouds of 8192..16384 points also keep their kd-tree ordering state (hg_knn_self_temporal_order_f32,
    see _TemporalOrders).  The loss and its gradient are the same bits either way; the states are per (batch shape,
    device) and replay-safe (the kernels update them in place)."""

    def __init__(self, k=5, alpha=1.05):
        super(KNNDist, self).__init__()
        self.k = k
        self.alpha = alpha
        self.temporal = False
        self._state = {}
        self._orders = {}

    def temporal_seeds(self, on=True):
        self.temporal = bool(on)
        self._state.clear()
        self._orders = {}
        return self

    def forward(self, pc, weights=None, batch_avg=True):
        """pc: [B, K, 3] or [B, 3, K] (dist_utils.py:145-147 treats shape[1] == 3 as channel-first)."""
        B = pc.shape[0]
        if pc.shape[1] == 3:
            pc = pc.transpose(2, 1)  # kernels are point-major
        state, valid, order = None, False, None
        # (getattr: install.patch_reference() binds this forward to the REFERENCE's KNNDist class, whose __init__ knows
        # nothing of the temporal state)
        if getattr(self, "temporal", False) and pc.is_cuda and pc.shape[2] == 3:
            key = (tuple(pc.shape), pc.device)
            valid = key in self._state
            if not valid:
                self._state[key] = torch.empty((pc.shape[0], pc.shape[1], self.k + 1), dtype=torch.int32, device=pc.device)
            state = self._state[key]
            order = _order(self._orders, "adv", pc)
        loss = F.knn_outlier_loss(pc, self.k, self.alpha, state, valid, order)  # [B]
        return _finish(loss, _weights(weights, B, loss.device), batch_avg)


class ChamferkNNDist(nn.Module):
    def __init__(self, chamfer_method='adv2ori', knn_k=5, knn_alpha=1.05, chamfer_weight=5., knn_weight=3.):
        super(ChamferkNNDist, self).__init__()
        self.chamfer_dist = ChamferDist(method=chamfer_method)
        self.knn_dist = KNNDist(k=knn_k, alpha=knn_alpha)
        self.w1 = chamfer_weight
        self.w2 = knn_weight

    def temporal_seeds(self, on=True):
        """Both terms: see KNNDist.temporal_seeds and ChamferDist.temporal_seeds.  The two terms share one ordering
        state of `adv`: forward runs them one after the other on the current stream, so the kNN term refits the
        ordering the Chamfer term has just refit or rebuilt."""
        self.chamfer_dist.temporal_seeds(on)
        self.knn_dist.temporal_seeds(on)
        self.knn_dist._orders = self.chamfer_dist._orders
        return self

    def forward(self, adv_pc, ori_pc, weights=None, batch_avg=True):
        chamfer_loss = self.chamfer_dist(adv_pc, ori_pc, weights=weights, batch_avg=batch_avg)
        knn_loss = self.knn_dist(adv_pc, weights=weights, batch_avg=batch_avg)
        loss = chamfer_loss * self.w1 + knn_loss * self.w2
        return loss
