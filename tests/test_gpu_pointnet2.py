"""Parity of the nine pointnet2_ops kernels against (a) the CPU oracle's restatement of the reference CUDA
kernels and (b), when oracle/_ref holds the reference's own kernels compiled for sm_100, those kernels run on
the same GPU.  Indices and gathered values bit-exact; scatter gradients 1e-5 (the reference sums them with
float atomics in arbitrary order, ours in a fixed order)."""
import importlib.util
import os
import warnings

import numpy as np
import pytest
import torch

from util_inputs import clouds, normwise

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def ext():
    from hitgeom.pointnet2_ops import _ext

    return _ext


@pytest.fixture(scope="module")
def ref_ext():
    """The reference's own `_ext`, compiled unmodified for sm_100 by oracle/build_ref.py (None if absent)."""
    so = os.path.join(ROOT, "oracle", "_ref", "_ext_ref.so")
    if not os.path.exists(so):
        warnings.warn("oracle/_ref/_ext_ref.so is not built (HITADV_REFERENCE=<checkout> python oracle/build_ref.py): "
                      "these tests compare with the oracle and the stored reference-kernel outputs only")
        return None
    spec = importlib.util.spec_from_file_location("_ext_ref", so)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


CASES = [(3, 1024, 51, "surface"), (2, 1024, 512, "gauss"), (2, 512, 128, "surface"), (4, 100, 17, "gauss"),
         (1, 4096, 64, "surface"), (2, 31, 31, "gauss"), (1, 600, 600, "gauss")]


@pytest.mark.parametrize("B,N,m,kind", CASES)
def test_fps(oracle, ext, ref_ext, B, N, m, kind):
    xyz = clouds(B, N, 400 + N, kind)
    out = ext.furthest_point_sampling(gpu(xyz), m)
    assert out.dtype == torch.int32 and tuple(out.shape) == (B, m)
    assert np.array_equal(out.cpu().numpy(), oracle.p2_fps(xyz, m))
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.furthest_point_sampling(gpu(xyz), m))


def test_fps_ties_and_origin(oracle, ext, ref_ext):
    """Exact duplicates (ties in the running distance) and points inside the 1e-3 origin ball."""
    xyz = clouds(2, 512, 9, "surface")
    xyz[:, 256:] = xyz[:, :256]  # every point twice -> ties everywhere
    xyz[:, 5] = 0.0
    out = ext.furthest_point_sampling(gpu(xyz), 300)
    assert np.array_equal(out.cpu().numpy(), oracle.p2_fps(xyz, 300))
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.furthest_point_sampling(gpu(xyz), 300))


@pytest.mark.parametrize("B,N,M,r,ns", [(3, 1024, 51, 0.126, 16), (2, 1024, 512, 0.2, 32), (2, 512, 128, 0.4, 64),
                                        (2, 1024, 51, 0.219, 49), (1, 300, 40, 0.01, 8), (2, 77, 13, 5.0, 100)])
def test_ball_query(oracle, ext, ref_ext, B, N, M, r, ns):
    xyz = clouds(B, N, 500 + N, "surface")
    new_xyz = xyz[:, :M].copy()
    new_xyz[:, -1] = 10.0  # a centre with an empty ball: the row stays zero
    out = ext.ball_query(gpu(new_xyz), gpu(xyz), r, ns)
    assert out.dtype == torch.int32
    assert np.array_equal(out.cpu().numpy(), oracle.p2_ball_query(new_xyz, xyz, r, ns))
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.ball_query(gpu(new_xyz), gpu(xyz), r, ns))


@pytest.mark.parametrize("B,C,N,M", [(3, 3, 1024, 51), (2, 64, 512, 128), (1, 1, 10, 40)])
def test_gather_and_grad(oracle, ext, ref_ext, B, C, N, M):
    rng = np.random.default_rng(1)
    pts = rng.standard_normal((B, C, N)).astype(np.float32)
    idx = rng.integers(0, N, (B, M)).astype(np.int32)
    idx[:, : M // 2] = idx[:, M // 2 : M // 2 * 2]  # repeated indices -> the grad really accumulates
    go = rng.standard_normal((B, C, M)).astype(np.float32)
    out = ext.gather_points(gpu(pts), gpu(idx))
    assert np.array_equal(out.cpu().numpy(), oracle.p2_gather(pts, idx))
    gr = ext.gather_points_grad(gpu(go), gpu(idx), N)
    assert normwise(gr.cpu().numpy(), oracle.p2_gather_grad(go, idx, N)) < 1e-6
    assert torch.equal(gr, ext.gather_points_grad(gpu(go), gpu(idx), N))  # deterministic
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.gather_points(gpu(pts), gpu(idx)))
        assert normwise(gr.cpu().numpy(), ref_ext.gather_points_grad(gpu(go), gpu(idx), N).cpu().numpy()) < 1e-5


@pytest.mark.parametrize("B,C,N,S,ns", [(3, 3, 1024, 51, 16), (2, 131, 512, 128, 64), (2, 3, 1024, 512, 32)])
def test_group_and_grad(oracle, ext, ref_ext, B, C, N, S, ns):
    rng = np.random.default_rng(2)
    xyz = clouds(B, N, 600 + N, "surface")
    idx = oracle.p2_ball_query(xyz[:, :S].copy(), xyz, 0.2, ns)  # realistic: heavy repetition from padding
    pts = rng.standard_normal((B, C, N)).astype(np.float32)
    go = rng.standard_normal((B, C, S, ns)).astype(np.float32)
    out = ext.group_points(gpu(pts), gpu(idx))
    assert np.array_equal(out.cpu().numpy(), oracle.p2_group(pts, idx))
    gr = ext.group_points_grad(gpu(go), gpu(idx), N)
    assert normwise(gr.cpu().numpy(), oracle.p2_group_grad(go, idx, N)) < 1e-5
    assert torch.equal(gr, ext.group_points_grad(gpu(go), gpu(idx), N))
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.group_points(gpu(pts), gpu(idx)))
        assert normwise(gr.cpu().numpy(), ref_ext.group_points_grad(gpu(go), gpu(idx), N).cpu().numpy()) < 1e-5


@pytest.mark.parametrize("B,n,m,c", [(2, 1024, 256, 64), (3, 100, 2, 5), (1, 700, 513, 3)])
def test_three_nn_and_interpolate(oracle, ext, ref_ext, B, n, m, c):
    rng = np.random.default_rng(3)
    unknown = clouds(B, n, 700 + n, "surface")
    known = clouds(B, m, 800 + m, "surface")
    d2, idx = ext.three_nn(gpu(unknown), gpu(known))
    od, oi = oracle.p2_three_nn(unknown, known)
    assert np.array_equal(d2.cpu().numpy(), od) and np.array_equal(idx.cpu().numpy(), oi)
    w = rng.random((B, n, 3)).astype(np.float32)
    w /= w.sum(-1, keepdims=True)
    pts = rng.standard_normal((B, c, m)).astype(np.float32)
    out = ext.three_interpolate(gpu(pts), idx, gpu(w))
    assert np.array_equal(out.cpu().numpy(), oracle.p2_three_interpolate(pts, oi, w))
    go = rng.standard_normal((B, c, n)).astype(np.float32)
    gr = ext.three_interpolate_grad(gpu(go), idx, gpu(w), m)
    assert normwise(gr.cpu().numpy(), oracle.p2_three_interpolate_grad(go, oi, w, m)) < 1e-5
    if ref_ext is not None:
        rd2, ridx = ref_ext.three_nn(gpu(unknown), gpu(known))
        assert torch.equal(d2, rd2) and torch.equal(idx, ridx)
        assert torch.equal(out, ref_ext.three_interpolate(gpu(pts), idx, gpu(w)))
        assert normwise(gr.cpu().numpy(), ref_ext.three_interpolate_grad(gpu(go), idx, gpu(w), m).cpu().numpy()) < 1e-5


def test_kernels_match_reference_kernel_golden(golden, ext):
    """The same kernels against stored outputs of the reference's own kernels on a B200
    (tests/golden/pointnet2_ref.npz, tests/golden/make_golden_gpu.py): bit-exact, without a build of the reference."""
    g = golden("pointnet2_ref")
    for tag in "abc":
        ref = g[f"fps_{tag}_idx"]
        assert np.array_equal(ext.furthest_point_sampling(gpu(g[f"fps_{tag}_xyz"]), ref.shape[1]).cpu().numpy(), ref), tag
    xyz, new_xyz = g["bq_xyz"], g["bq_new_xyz"]
    assert np.array_equal(ext.furthest_point_sampling(gpu(xyz), 51).cpu().numpy(), g["bq_fps"])
    gathered = ext.gather_points(gpu(xyz.transpose(0, 2, 1)), gpu(g["bq_fps"]))
    assert np.array_equal(gathered.cpu().numpy().transpose(0, 2, 1), new_xyz)
    for key in g.files:
        if key.startswith("bq_r"):
            r, ns = float(key.split("_")[1][1:]), int(key.split("_")[2][2:])
            assert np.array_equal(ext.ball_query(gpu(new_xyz), gpu(xyz), r, ns).cpu().numpy(), g[key]), key
    assert np.array_equal(ext.group_points(gpu(g["grp_points"]), gpu(g["bq_r0.2_ns32"])).cpu().numpy(), g["grp_out"])
    d2, idx = ext.three_nn(gpu(g["nn_unknown"]), gpu(g["nn_known"]))
    assert np.array_equal(d2.cpu().numpy(), g["nn_dist2"]) and np.array_equal(idx.cpu().numpy(), g["nn_idx"])
    out = ext.three_interpolate(gpu(g["ti_feats"]), gpu(g["nn_idx"]), gpu(g["ti_w"]))
    assert np.array_equal(out.cpu().numpy(), g["ti_out"])


def test_autograd_wrappers_and_query_and_group(oracle):
    """The autograd layer: same public names / signatures as pointnet2_ops.pointnet2_utils."""
    from hitgeom.pointnet2_ops import pointnet2_utils as pu

    xyz_np = clouds(2, 512, 42, "surface")
    xyz = gpu(xyz_np)
    fps = pu.furthest_point_sample(xyz, 64)
    assert not fps.requires_grad and fps.dtype == torch.int32
    feats = torch.randn(2, 8, 512, device="cuda", requires_grad=True)
    new_xyz = pu.gather_operation(xyz.transpose(1, 2).contiguous(), fps).transpose(1, 2).contiguous()
    grouper = pu.QueryAndGroup(0.3, 16, use_xyz=True)
    out = grouper(xyz, new_xyz, feats)
    assert tuple(out.shape) == (2, 11, 64, 16)
    out.sum().backward()
    idx = oracle.p2_ball_query(new_xyz.cpu().numpy(), xyz_np, 0.3, 16)
    expect = oracle.p2_group_grad(np.ones((2, 8, 64, 16), np.float32), idx, 512)
    assert normwise(feats.grad.cpu().numpy(), expect) < 1e-6
    dist, idx3 = pu.three_nn(xyz, new_xyz)
    w = torch.full((2, 512, 3), 1.0 / 3, device="cuda")
    f2 = torch.randn(2, 4, 64, device="cuda", requires_grad=True)
    pu.three_interpolate(f2, idx3, w).sum().backward()
    assert f2.grad is not None and torch.isfinite(f2.grad).all()
    ga = pu.GroupAll()(xyz, None, feats)
    assert tuple(ga.shape) == (2, 11, 1, 512)


def test_ext_rejects_bad_input(ext):
    with pytest.raises(RuntimeError):
        ext.furthest_point_sampling(torch.zeros(1, 8, 3), 2)  # CPU not supported
    with pytest.raises(RuntimeError):
        ext.gather_points(torch.zeros(1, 3, 8, device="cuda"), torch.zeros(1, 2, device="cuda", dtype=torch.int64))
    with pytest.raises(RuntimeError):
        ext.group_points(torch.zeros(1, 3, 8, device="cuda").transpose(1, 2), torch.zeros(1, 2, 2, device="cuda", dtype=torch.int32))


def test_uniform_loss_pipeline_vs_oracle(oracle):
    """The op sequence of the one in-repo pointnet2_ops caller, `uniform_loss` (FGM/GeoA3_args.py:258-302): for five
    ball sizes, FPS(5% of n) -> gather -> ball_query -> group -> kNN inside every ball -> the uniformity statistic.
    Every index tensor bit-exact against the oracle's composition; the final scalar to 1e-5."""
    import math

    from hitgeom.pointnet2_ops import pointnet2_utils as pu
    from hitgeom.pytorch3d_ops import knn_points

    B, n = 3, 1024
    pc_np = clouds(B, n, 321, "surface")
    pc = gpu(pc_np)
    npoint = int(n * 0.05)
    loss, loss_ref = 0.0, 0.0
    for p in [0.004, 0.006, 0.008, 0.010, 0.012]:
        p4 = p * 4
        nsample, r = int(n * p4), math.sqrt(p4 * 1.0)
        expect_len = math.sqrt(math.pi * p4 / nsample)
        flipped = pc.transpose(1, 2).contiguous()
        fps = pu.furthest_point_sample(pc, npoint)
        new_xyz = pu.gather_operation(flipped, fps).transpose(1, 2).contiguous()
        idx = pu.ball_query(r, nsample, pc, new_xyz)
        grouped = pu.grouping_operation(flipped, idx).permute(0, 2, 3, 1).contiguous()  # [B,npoint,nsample,3]
        grouped = torch.cat(torch.unbind(grouped, dim=1), dim=0)  # [B*npoint,nsample,3]
        knn = knn_points(grouped, grouped, K=3)
        d = torch.sqrt(torch.abs(knn.dists[:, :, 1:]) + 1e-12).mean(dim=-1)
        loss = loss + (((d - expect_len) ** 2 / (expect_len + 1e-12)).reshape(-1).mean() * (p4 * 100) ** 2).item()
        # oracle composition
        ofps = oracle.p2_fps(pc_np, npoint)
        onew = oracle.p2_gather(pc_np.transpose(0, 2, 1), ofps).transpose(0, 2, 1)
        oidx = oracle.p2_ball_query(np.ascontiguousarray(onew), pc_np, np.float32(r), nsample)
        ogrp = oracle.p2_group(pc_np.transpose(0, 2, 1), oidx).transpose(0, 2, 3, 1)
        ogrp = np.concatenate([ogrp[:, s] for s in range(npoint)], axis=0)
        od, oi = oracle.knn_points(ogrp, ogrp, 3, threads=4)
        assert np.array_equal(fps.cpu().numpy(), ofps) and np.array_equal(idx.cpu().numpy(), oidx)
        assert np.array_equal(grouped.cpu().numpy(), ogrp)
        assert np.array_equal(knn.idx.cpu().numpy(), oi) and np.array_equal(knn.dists.cpu().numpy(), od)
        dd = np.sqrt(np.abs(od[:, :, 1:].astype(np.float64)) + 1e-12).mean(-1)
        loss_ref += ((dd - expect_len) ** 2 / (expect_len + 1e-12)).reshape(-1).mean() * (p4 * 100) ** 2
    assert abs(loss - loss_ref) <= 1e-5 * abs(loss_ref)


def test_fps_large_cloud(oracle, ext, ref_ext):
    """16384-point clouds (config 5 size): the 1024-thread variant of the FPS kernel."""
    xyz = clouds(2, 16384, 1616, "surface")
    out = ext.furthest_point_sampling(gpu(xyz), 96)
    assert np.array_equal(out.cpu().numpy(), oracle.p2_fps(xyz, 96))
    if ref_ext is not None:
        assert torch.equal(out, ref_ext.furthest_point_sampling(gpu(xyz), 96))
    xyz5 = clouds(1, 5000, 55, "gauss")
    assert np.array_equal(ext.furthest_point_sampling(gpu(xyz5), 40).cpu().numpy(), oracle.p2_fps(xyz5, 40))
