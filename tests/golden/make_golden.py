"""Generate tests/golden/*.npz by running the UNMODIFIED reference (imported from /root/reference) on seeded
synthetic inputs.  Run in the build container only:  python tests/golden/make_golden.py

The reference ships no golden vectors or tests of its own (SURVEY.md section 4), so these fixtures -- outputs of
the reference's torch path on CPU, torch 2.11 -- are what pins the oracle (tests/test_oracle_golden.py) and,
through it, the CUDA kernels.  Each fixture stores the inputs next to the outputs so the tests never need
/root/reference.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _refload  # noqa: E402


def clouds(B, N, seed, kind="gauss"):
    """Synthetic clouds per SURVEY.md section 8d: unit-ball normalised like Dataset/ModelNet.py:12-17."""
    g = torch.Generator().manual_seed(seed)
    if kind == "gauss":
        x = torch.randn(B, N, 3, generator=g)
    else:  # surface-like: a few planes + spheres, 1% exact duplicates, a few near-origin points
        x = torch.randn(B, N, 3, generator=g)
        x[:, : N // 2] = x[:, : N // 2] / x[:, : N // 2].norm(dim=-1, keepdim=True)
        x[:, N // 2 :, 2] = 0.25
        ndup = max(1, N // 100)
        src = torch.randint(0, N, (B, ndup), generator=g)
        dst = torch.randint(0, N, (B, ndup), generator=g)
        for b in range(B):
            x[b, dst[b]] = x[b, src[b]]
    x = x - x.mean(dim=1, keepdim=True)
    x = x / x.norm(dim=-1).amax(dim=1)[:, None, None]
    if kind != "gauss":
        x[:, :3] = x[:, :3] * 1e-3  # near-origin points (FPS origin-skip, sampling_gpu.cu:101)
    return x.contiguous()


def jitter(x, seed, sigma=0.01, clip=0.05):
    g = torch.Generator().manual_seed(seed)
    return (x + torch.clamp(sigma * torch.randn(x.shape, generator=g), -clip, clip)).contiguous()


def save(name, **arrs):
    out = {}
    for k, v in arrs.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        out[k] = np.asarray(v)
    path = os.path.join(HERE, name + ".npz")
    np.savez_compressed(path, **out)
    print(f"{name}: {os.path.getsize(path) / 1024:.1f} KiB")


def set_distance_cases(ref):
    sd = ref.set_distance
    for name, B, N1, N2, kind in [("setdist_eq", 3, 256, 256, "gauss"), ("setdist_ragged", 4, 96, 160, "gauss"),
                                  ("setdist_dups", 2, 200, 200, "surface")]:
        gts = clouds(B, N2, 1234, kind)
        if N1 == N2:
            preds = jitter(gts, 99)
        else:
            preds = jitter(clouds(B, N1, 77, kind), 99)
        out = {"gts": gts, "preds": preds}
        P = sd.chamfer.batch_pairwise_dist(gts, preds)
        m1, a1 = torch.min(P, 1)
        m2, a2 = torch.min(P, 2)
        out.update(min1=m1, arg1=a1, min2=m2, arg2=a2)
        if B * N1 * N2 <= 3 * 256 * 256:
            out["P"] = P
        for fn, tag in [(sd.chamfer, "ch"), (sd.hausdorff, "hd")]:
            for which in (0, 1):
                p = preds.clone().requires_grad_()
                g = gts.clone().requires_grad_()
                losses = fn(p, g)
                w = torch.linspace(0.5, 1.5, B)
                (losses[which] * w).sum().backward()
                out[f"{tag}_loss{which + 1}"] = losses[which]
                out[f"{tag}_grad_preds{which + 1}"] = p.grad
                out[f"{tag}_grad_gts{which + 1}"] = g.grad
        out["w"] = torch.linspace(0.5, 1.5, B)
        save(name, **out)

    # R3: channel-first input as HiT_ADV.py:229-231 passes it -> a 3x3 matrix over coordinate rows, inner dim K
    B, K = 4, 1024
    ori = clouds(B, K, 5).transpose(1, 2).contiguous()  # [B,3,K]
    adv = jitter(ori, 6)
    p = adv.clone().requires_grad_()
    P = sd.chamfer.batch_pairwise_dist(ori, adv)
    l1, l2 = sd.chamfer(p, ori)
    w = torch.linspace(0.5, 1.5, B)
    ((l1 + 2 * l2) * w).sum().backward()
    save("setdist_channel_first", gts=ori, preds=adv, P=P, ch_loss1=l1, ch_loss2=l2, grad_preds=p.grad, w=w)


def loss_class_cases(ref):
    du = ref.dist_utils
    B, K = 4, 256
    ori = clouds(B, K, 11)
    adv = jitter(ori, 12)
    w = torch.tensor([1.0, 0.25, 2.0, 0.0], dtype=torch.float64)  # CW/Perturb.py:148-150 passes float64 weights
    out = {"ori": ori, "adv": adv, "w": w}
    for cls, tag in [(du.ChamferDist, "chamfer"), (du.HausdorffDist, "hausdorff")]:
        for method in ("adv2ori", "ori2adv", "both"):
            for wt, wtag in [(None, "now"), (w, "w")]:
                for avg in (True, False):
                    a = adv.clone().requires_grad_()
                    loss = cls(method=method)(a, ori, weights=wt, batch_avg=avg)
                    loss.sum().backward()
                    key = f"{tag}_{method}_{wtag}_{'avg' if avg else 'vec'}"
                    out[key] = loss
                    out[key + "_grad"] = a.grad
    for k, alpha in [(5, 1.05), (4, 1.05), (8, 0.5)]:
        for layout in ("BK3", "B3K"):
            for wt, wtag in [(None, "now"), (w, "w")]:
                a = adv.clone().requires_grad_()
                inp = a if layout == "BK3" else a.transpose(1, 2).contiguous()
                if layout == "B3K":
                    a = inp.detach().clone().requires_grad_()
                    inp = a
                loss = du.KNNDist(k=k, alpha=alpha)(inp, weights=wt, batch_avg=False)
                loss.sum().backward()
                key = f"knn_k{k}_{layout}_{wtag}"
                out[key] = loss
                out[key + "_grad"] = a.grad
    # internals of KNNDist for k=5 (dist_utils.py:148-166) so the oracle's intermediate tensors are pinned too; the
    # [B,K,K] matrix itself is not stored (no test reads it, and it alone would take the file past 1 MB)
    pc = adv.transpose(2, 1)
    inner = -2.0 * torch.matmul(pc.transpose(2, 1), pc)
    xx = torch.sum(pc ** 2, dim=1, keepdim=True)
    dist = xx + inner + xx.transpose(2, 1)
    neg_value, idx = (-dist).topk(k=6, dim=-1)
    out.update(knn_topk_vals=-neg_value, knn_topk_idx=idx)
    a = adv.clone().requires_grad_()
    loss = du.ChamferkNNDist()(a, ori, weights=w, batch_avg=True)
    loss.backward()
    out.update(chamferknn=loss, chamferknn_grad=a.grad)
    a = adv.clone().requires_grad_()
    loss = du.ChamferkNNDist(chamfer_method="both", knn_k=4, knn_alpha=1.1, chamfer_weight=2.0, knn_weight=0.5)(
        a, ori, batch_avg=False)
    loss.sum().backward()
    out.update(chamferknn2=loss, chamferknn2_grad=a.grad)
    save("loss_classes", **out)


def seam_cases(ref):
    pu = ref.pn2_utils
    B, N = 3, 512
    xyz = clouds(B, N, 21, "surface")
    out = {"xyz": xyz}
    torch.manual_seed(7)
    start = torch.randint(0, N, (B,), dtype=torch.long)
    torch.manual_seed(7)
    fps = pu.farthest_point_sample(xyz, 64)
    assert torch.equal(fps[:, 0], start)
    out.update(fps_start=start, fps_idx=fps)
    new_xyz = pu.index_points(xyz, fps)
    out["new_xyz"] = new_xyz
    out["sqdist"] = pu.square_distance(new_xyz, xyz)
    for r, ns in [(0.2, 32), (0.4, 64), (0.15, 16), (0.05, 8)]:
        out[f"ball_r{r}_ns{ns}"] = pu.query_ball_point(r, ns, xyz, new_xyz)
    idx = out["ball_r0.2_ns32"]
    out["index_points_grouped"] = pu.index_points(xyz, idx)
    save("torch_seams", **out)


def dgcnn_cases(ref):
    knn = ref.dgcnn.knn
    out = {}
    x3 = clouds(2, 256, 31).transpose(1, 2).contiguous()  # [B,3,N]
    out.update(x3=x3, idx3_k20=knn(x3, 20), idx3_k5=knn(x3, 5))
    for C in (64, 128):
        g = torch.Generator().manual_seed(40 + C)
        x = torch.randn(2, C, 192, generator=g)
        inner = -2 * torch.matmul(x.transpose(2, 1), x)
        xx = torch.sum(x ** 2, dim=1, keepdim=True)
        pw = -xx - inner - xx.transpose(2, 1)
        out.update({f"x{C}": x, f"idx{C}_k20": knn(x, 20), f"pw{C}": pw})
    save("dgcnn_knn", **out)


if __name__ == "__main__":
    torch.set_num_threads(8)
    ref = _refload.load()
    set_distance_cases(ref)
    loss_class_cases(ref)
    seam_cases(ref)
    dgcnn_cases(ref)
