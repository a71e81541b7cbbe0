"""Kernel-backed versions of the torch-level geometry functions the victims call inside forward:

  model/pointnet2_utils.py:19-40   square_distance(src, dst)
  model/pointnet2_utils.py:43-60   index_points(points, idx)                 (differentiable in points)
  model/pointnet2_utils.py:63-84   farthest_point_sample(xyz, npoint)        (random start: torch.randint)
  model/pointnet2_utils.py:87-107  query_ball_point(radius, nsample, xyz, new_xyz)
  model/dgcnn_cls.py:7-13          knn(x, k)                                 (x is channel-major [B,C,N])
  model/dgcnn_cls.py:16-43         get_graph_feature(x, k=20, idx=None, dim9=False)  (differentiable in x)

Same signatures, dtypes (int64 indices) and semantics, so `hitgeom.install()` can rebind them into the
reference's module globals and PointNet++ SSG / DGCNN run unchanged (`sample_and_group` and
`get_graph_feature` look the names up at call time).
"""
import torch

from . import functional as F


class _SquareDistanceFn(torch.autograd.Function):
    """The reference's square_distance is plain torch (matmul + sums) and therefore differentiable:
    PointNetFeaturePropagation differentiates its interpolation weights through it (model/pointnet2_utils.py:297-303).
    Forward = the kernel (reference rounding order); backward = what autograd derives for d[n,m] = |s_n - t_m|^2:
    grad_src[n] = 2 s_n sum_m g[n,m] - 2 (g @ dst)[n], grad_dst[m] = 2 t_m sum_n g[n,m] - 2 (g^T @ src)[m]."""

    @staticmethod
    def forward(ctx, src, dst):
        ctx.save_for_backward(src, dst)
        return F.square_distance(src.detach().contiguous(), dst.detach().contiguous())

    @staticmethod
    def backward(ctx, g):
        src, dst = ctx.saved_tensors
        gs = gd = None
        if ctx.needs_input_grad[0]:
            gs = 2.0 * (src * g.sum(dim=2, keepdim=True) - torch.bmm(g, dst))
        if ctx.needs_input_grad[1]:
            gd = 2.0 * (dst * g.sum(dim=1).unsqueeze(2) - torch.bmm(g.transpose(1, 2), src))
        return gs, gd


def square_distance(src, dst):
    """[B,N,C] x [B,M,C] -> [B,N,M] = ((-2 src.dst) + |src|^2) + |dst|^2, the reference's rounding order;
    differentiable in both arguments."""
    if src.requires_grad or dst.requires_grad:
        return _SquareDistanceFn.apply(src, dst)
    return F.square_distance(src.contiguous(), dst.contiguous())


def index_points(points, idx):
    """points [B,N,C], idx [B,S] or [B,S,ns] (int64) -> [B,S,C] / [B,S,ns,C]."""
    B = points.shape[0]
    flat = idx.reshape(B, -1).contiguous()
    if flat.dtype != torch.int64:
        flat = flat.long()
    out = F.IndexPointsFn.apply(points, flat)
    return out.view(*idx.shape, points.shape[-1])


def farthest_point_sample(xyz, npoint):
    """xyz [B,N,3] -> centroids [B,npoint] int64.  The start index is drawn exactly as the reference does
    (`torch.randint(0, N, (B,))` on the CPU generator, pointnet2_utils.py:75), so a seeded run reproduces it."""
    device = xyz.device
    B, N, C = xyz.shape
    farthest = torch.randint(0, N, (B,), dtype=torch.long).to(device)
    return F.fps_torch(xyz.detach().contiguous(), int(npoint), farthest)


def query_ball_point(radius, nsample, xyz, new_xyz):
    """xyz [B,N,3], new_xyz [B,S,3] -> group_idx [B,S,nsample] int64 (ascending, padded with the first hit)."""
    return F.query_ball_torch(radius, int(nsample), xyz.detach().contiguous(), new_xyz.detach().contiguous())


def knn(x, k):
    """DGCNN kNN: x [B,C,N] -> idx [B,N,k] int64, the k largest of -||x_i - x_j||^2 (self included); 1 <= k <= 64
    for every C (DGCNN's k = 20 and k = 40 included)."""
    pc = x.detach().transpose(2, 1).contiguous()  # kernels are point-major
    _, idx = F.knn_self(pc, int(k), want_vals=False)
    return idx.long()


def get_graph_feature(x, k=20, idx=None, dim9=False):
    """x [B,C,N] -> edge features [B,2C,N,k] = cat(x[idx] - x, x) (dgcnn_cls.py:16-43), one kernel instead of
    gather + repeat + cat + permute().contiguous(); kNN on the features (or on channels 6: when `dim9`)."""
    batch_size, num_points = x.size(0), x.size(2)
    x = x.view(batch_size, -1, num_points)
    if idx is None:
        idx = knn(x if not dim9 else x[:, 6:], k=k)
    return F.edge_feature(x, idx)
