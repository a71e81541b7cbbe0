"""Parity of the CUDA Chamfer / Hausdorff path (through the Python mirror -> C ABI) against the golden
vectors of the reference and against the CPU oracle.  Bar: min values and argmin indices BIT-EXACT;
losses within 1e-6 relative; gradients within 1e-5 norm-wise per sample."""
import numpy as np
import pytest
import torch

from util_inputs import clouds, jitter, normwise

pytestmark = pytest.mark.gpu


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def F():
    from hitgeom import functional

    return functional


@pytest.fixture(autouse=True, params=["exact-tracker", "exact-tracker-gather-finish"])
def _tracker(request):
    """Every test of this module runs twice: with the default distance pass (5-operation exact tracker; clouds that fit
    in shared memory finish in nn_bidir_d3_finish_small_kernel), and with the general gather finish kernel forced for
    small clouds too (hg_tune("small_fused", 1)).  Both must give the reference's bits."""
    from hitgeom._lib import lib

    lib().hg_tune(b"small_fused", 1 if request.param == "exact-tracker-gather-finish" else 0)
    yield request.param
    lib().hg_tune(b"small_fused", 0)


@pytest.mark.parametrize("name", ["setdist_eq", "setdist_ragged", "setdist_dups"])
@pytest.mark.parametrize("T", [0, 8, 16])
def test_nn_bidir_golden(golden, F, name, T):
    g = golden(name)
    F.tune_nn_bidir(T, 0)
    try:
        m1, a1, m2, a2 = F.nn_bidir(gpu(g["gts"]), gpu(g["preds"]))
    finally:
        F.tune_nn_bidir(0, 0)
    assert np.array_equal(m1.cpu().numpy(), g["min1"])
    assert np.array_equal(m2.cpu().numpy(), g["min2"])
    assert np.array_equal(a1.cpu().numpy(), g["arg1"])
    assert np.array_equal(a2.cpu().numpy(), g["arg2"])


@pytest.mark.parametrize("B,N2,N1,kind", [(1, 1, 1, "gauss"), (2, 7, 5, "gauss"), (3, 33, 129, "gauss"),
                                          (2, 513, 511, "surface"), (2, 1024, 1024, "surface"),
                                          (1, 3000, 2049, "gauss"), (5, 64, 640, "surface")])
@pytest.mark.parametrize("T,RB", [(0, 0), (8, 8), (16, 24), (16, 256)])
def test_nn_bidir_vs_oracle(oracle, F, B, N2, N1, kind, T, RB):
    gts = clouds(B, max(N2, 2), 100 + N2, kind)[:, :N2].copy()  # (a 1-point cloud cannot be normalised)
    preds = jitter(clouds(B, max(N1, 2), 100 + N2, kind)[:, :N1], 7) if N1 != N2 else jitter(gts, 7)
    F.tune_nn_bidir(T, RB)
    try:
        m1, a1, m2, a2 = F.nn_bidir(gpu(gts), gpu(preds))
    finally:
        F.tune_nn_bidir(0, 0)
    o1, oa1, o2, oa2 = oracle.nn_bidir(gts, preds, threads=4)
    assert np.array_equal(m1.cpu().numpy(), o1) and np.array_equal(m2.cpu().numpy(), o2)
    assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2)


def test_nn_bidir_identical_clouds_ties(oracle, F):
    """adv == ori and many exact duplicates: every tie must resolve to the first index like torch.min."""
    gts = clouds(2, 300, 5, "surface")
    gts[:, 100:200] = gts[:, 0:100]
    m1, a1, m2, a2 = F.nn_bidir(gpu(gts), gpu(gts.copy()))
    o1, oa1, o2, oa2 = oracle.nn_bidir(gts, gts)
    assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2)
    assert np.array_equal(m1.cpu().numpy(), o1) and np.array_equal(m2.cpu().numpy(), o2)


@pytest.mark.parametrize("name", ["setdist_eq", "setdist_ragged", "setdist_dups"])
@pytest.mark.parametrize("tag", ["ch", "hd"])
def test_losses_and_grads_golden(golden, name, tag):
    from hitgeom.set_distance import chamfer, hausdorff

    g = golden(name)
    fn = chamfer if tag == "ch" else hausdorff
    w = gpu(g["w"])
    for which in (0, 1):
        p = gpu(g["preds"]).requires_grad_()
        x = gpu(g["gts"]).requires_grad_()
        losses = fn(p, x)
        (losses[which] * w).sum().backward()
        ref = g[f"{tag}_loss{which + 1}"]
        np.testing.assert_allclose(losses[which].detach().cpu().numpy(), ref, rtol=1e-6 if tag == "ch" else 0, atol=0)
        assert normwise(p.grad.cpu().numpy(), g[f"{tag}_grad_preds{which + 1}"]) < 1e-5
        assert normwise(x.grad.cpu().numpy(), g[f"{tag}_grad_gts{which + 1}"]) < 1e-5


def test_channel_first_degenerate(golden, oracle):
    """SURVEY.md R3: [B,3,K] inputs -> 3x3 matrix with inner dim K.  The CUDA generic-D kernel uses the same
    sequential FMA chain as the oracle (bit-exact vs oracle); vs the reference's MKL GEMM the difference is
    summation-order noise, bounded in ulps of the cancelling operands."""
    from hitgeom.set_distance import chamfer

    g = golden("setdist_channel_first")
    P = chamfer.batch_pairwise_dist(gpu(g["gts"]), gpu(g["preds"])).cpu().numpy()
    assert np.array_equal(P, oracle.pairwise_dist(g["gts"], g["preds"]))
    ulp = np.spacing(np.float32(np.abs(g["P"]).max()))
    assert np.abs(P - g["P"]).max() <= 32 * ulp
    p = gpu(g["preds"]).requires_grad_()
    l1, l2 = chamfer(p, gpu(g["gts"]))
    assert np.abs(l1.detach().cpu().numpy() - g["ch_loss1"]).max() <= 32 * ulp
    assert np.abs(l2.detach().cpu().numpy() - g["ch_loss2"]).max() <= 32 * ulp
    ((l1 + 2 * l2) * gpu(g["w"])).sum().backward()
    # gradient: same argmins as the reference here (3x3 with a clear diagonal) -> 1e-4 of the norm
    assert normwise(p.grad.cpu().numpy(), g["grad_preds"]) < 1e-4


def test_loss_classes_golden(golden):
    from hitgeom.dist_utils import ChamferDist, ChamferkNNDist, HausdorffDist

    g = golden("loss_classes")
    ori = gpu(g["ori"])
    w = torch.from_numpy(g["w"])  # float64 CPU tensor, as CW/Perturb.py:148-150 passes it
    for cls, tag in [(ChamferDist, "chamfer"), (HausdorffDist, "hausdorff")]:
        for method in ("adv2ori", "ori2adv", "both"):
            for wt, wtag in [(None, "now"), (w, "w")]:
                for avg in (True, False):
                    a = gpu(g["adv"]).requires_grad_()
                    loss = cls(method=method)(a, ori, weights=wt, batch_avg=avg)
                    loss.sum().backward()
                    key = f"{tag}_{method}_{wtag}_{'avg' if avg else 'vec'}"
                    np.testing.assert_allclose(loss.detach().cpu().numpy(), g[key], rtol=2e-6, atol=0, err_msg=key)
                    gr, ref = a.grad.cpu().numpy(), g[key + "_grad"]
                    assert np.abs(gr - ref).max() <= 1e-5 * np.abs(ref).max(), key
    a = gpu(g["adv"]).requires_grad_()
    loss = ChamferkNNDist()(a, ori, weights=w, batch_avg=True)
    loss.backward()
    np.testing.assert_allclose(loss.item(), g["chamferknn"], rtol=2e-6)
    assert np.abs(a.grad.cpu().numpy() - g["chamferknn_grad"]).max() <= 1e-5 * np.abs(g["chamferknn_grad"]).max()
    a = gpu(g["adv"]).requires_grad_()
    loss = ChamferkNNDist(chamfer_method="both", knn_k=4, knn_alpha=1.1, chamfer_weight=2.0, knn_weight=0.5)(
        a, ori, batch_avg=False)
    loss.sum().backward()
    np.testing.assert_allclose(loss.detach().cpu().numpy(), g["chamferknn2"], rtol=2e-6)
    assert normwise(a.grad.cpu().numpy(), g["chamferknn2_grad"]) < 1e-5


def test_config1_full_size_vs_oracle(oracle, F):
    """BASELINE config 1 shape: 388 x 1024 clouds vs jittered copies -- bit-exact against the oracle."""
    ori = clouds(388, 1024, 1234)
    adv = jitter(ori, 99)
    m1, a1, m2, a2 = F.nn_bidir(gpu(ori), gpu(adv))
    o1, oa1, o2, oa2 = oracle.nn_bidir(ori, adv, threads=oracle.host_threads())
    assert np.array_equal(m1.cpu().numpy(), o1) and np.array_equal(m2.cpu().numpy(), o2)
    assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2)


def test_large_cloud_properties(oracle, F):
    """Config 5 shape (16384 points per cloud).  (i) a cloud against itself: every min is attained at the point
    itself or an exact duplicate; (ii) min values are invariant under a permutation of preds and the returned
    index attains them (checked by re-evaluating the reference formula at the returned pairs); (iii) two full
    clouds bit-exact against the oracle (a few seconds of CPU)."""
    x = clouds(3, 16384, 77)
    xg = gpu(x)
    m1, a1, m2, a2 = F.nn_bidir(xg, xg.clone())
    a1c, a2c = a1.cpu().numpy(), a2.cpu().numpy()
    assert np.array_equal(x[np.arange(3)[:, None], a1c], x) and np.array_equal(x[np.arange(3)[:, None], a2c], x)
    perm = np.random.default_rng(0).permutation(16384)
    y = jitter(x, 3)
    yp = np.ascontiguousarray(y[:, perm])
    _, _, m2a, a2a = F.nn_bidir(xg, gpu(y))
    _, _, m2b, a2b = F.nn_bidir(xg, gpu(yp))
    assert np.array_equal(m2a.cpu().numpy(), m2b.cpu().numpy())
    picked = yp[np.arange(3)[:, None], a2b.cpu().numpy()]  # [3,N,3]: the pred each gt point was matched to
    P = oracle.pairwise_dist(x.reshape(-1, 1, 3), picked.reshape(-1, 1, 3)).reshape(3, -1)
    assert np.array_equal(P, m2b.cpu().numpy())
    o1, oa1, o2, oa2 = oracle.nn_bidir(x[:2], y[:2], threads=oracle.host_threads())
    r1, ra1, r2, ra2 = F.nn_bidir(gpu(x[:2]), gpu(y[:2]))
    assert np.array_equal(r1.cpu().numpy(), o1) and np.array_equal(r2.cpu().numpy(), o2)
    assert np.array_equal(ra1.cpu().numpy(), oa1) and np.array_equal(ra2.cpu().numpy(), oa2)


def test_errors_are_exceptions(F):
    from hitgeom import HitgeomError

    with pytest.raises(RuntimeError):
        F.nn_bidir(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3))  # CPU tensors
    with pytest.raises(RuntimeError):
        F.nn_bidir(torch.zeros(1, 4, 3, device="cuda").transpose(1, 2), torch.zeros(1, 4, 3, device="cuda"))
    with pytest.raises(RuntimeError):
        F.nn_bidir(torch.zeros(1, 4, 3, device="cuda", dtype=torch.float64), torch.zeros(1, 4, 3, device="cuda"))
    with pytest.raises((HitgeomError, RuntimeError)):
        F.knn_self(torch.zeros(1, 4, 3, device="cuda"), 9)  # k > K


def test_shared_distance_pass_is_transparent():
    """Inside `shared_distance_pass()` Chamfer + Hausdorff of the same pair run ONE distance pass; values and gradients
    are the bits of the unshared computation, and a modified cloud (version bump) is never served from the cache."""
    from hitgeom import _lib
    from hitgeom.dist_utils import ChamferDist, HausdorffDist, shared_distance_pass

    ori = gpu(clouds(4, 700, 3))
    adv = gpu(jitter(clouds(4, 700, 3), 8)).requires_grad_()
    cd, hd = ChamferDist(method="ori2adv"), HausdorffDist(method="adv2ori")

    def run(shared):
        adv.grad = None
        n0 = _lib.launch_count()
        if shared:
            with shared_distance_pass():
                loss = cd(adv, ori) + hd(adv, ori)
        else:
            loss = cd(adv, ori) + hd(adv, ori)
        launches = _lib.launch_count() - n0
        loss.backward()
        return loss.detach().clone(), adv.grad.clone(), launches

    l0, g0, n_plain = run(False)
    l1, g1, n_shared = run(True)
    assert torch.equal(l0, l1) and torch.equal(g0, g1)
    assert n_shared < n_plain
    with shared_distance_pass():
        a = cd(adv, ori)
        with torch.no_grad():
            adv.add_(0.01)  # in-place update (what an optimiser step does): bumps the version
        b = cd(adv, ori)
        assert a.item() != b.item()
    assert torch.equal(b.detach(), cd(adv, ori).detach())


def test_backward_with_hub_points_vs_oracle(oracle):
    """Degenerate clouds (ADVICE r1): thousands of sources sharing ONE nearest neighbour -- a collapsed adversarial
    cloud, or padding by repetition.  The reverse-map walk switches from selection (O(deg^2)) to a forward-map scan for
    in-degrees above 32; the gradient must still be the oracle's ascending-order sum and the call must return promptly."""
    import time

    from hitgeom import functional as F

    B, N = 2, 4096
    ori = clouds(B, N, 5)
    adv = jitter(ori, 6)
    adv[0, :] = adv[0, 0]          # cloud 0: the whole adversarial cloud collapsed onto one point
    adv[1, : N // 2] = adv[1, 7]   # cloud 1: half of it
    ori[1, N // 2:] = ori[1, 3]    # and half of the original cloud repeated
    o, a = torch.from_numpy(ori).cuda(), torch.from_numpy(adv).cuda()
    m1, a1, m2, a2 = F.nn_bidir(o, a)
    for mode in (0, 1):
        l1, l2, h1, h2 = F.set_loss(m1, m2, mode)
        g1 = torch.tensor([0.7, 1.3], device="cuda")
        g2 = torch.tensor([1.1, 0.4], device="cuda")
        torch.cuda.synchronize()
        t0 = time.time()
        gp, gg = F.set_loss_bwd(o, a, a1, a2, h1, h2, g1, g2, mode, True)
        torch.cuda.synchronize()
        assert time.time() - t0 < 2.0
        o1, oa1, o2, oa2 = oracle.nn_bidir(ori, adv)
        assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2)
        _, _, oh1, oh2 = oracle.set_loss(o1, o2, mode)
        wp, wg = oracle.set_loss_bwd(ori, adv, oa1, oa2, oh1, oh2, g1.cpu().numpy(), g2.cpu().numpy(), mode, want_gts=True)
        # a hub's gradient is an FP32 sum of thousands of terms: FMA contraction alone (nvcc fuses 2*(v-x) into the
        # accumulation, gcc does not) moves it by ~sqrt(deg) ulp, so the gate here is 1e-4, not the 1e-5 of regular clouds
        assert normwise(gp.cpu().numpy(), wp) < 1e-4 and normwise(gg.cpu().numpy(), wg) < 1e-4, mode


@pytest.mark.parametrize("case", ["dups across batches", "far from origin", "all equal", "lattice", "tiny spacings"])
def test_nn_bidir_ambiguous_inputs_vs_oracle(oracle, F, case):
    """Inputs full of ties and near-ties: exact duplicates spread over different 32-row batches and different lanes,
    clouds far from the origin (rounding of |p|^2 larger than the nearest-neighbour gaps), a cloud of identical points,
    an integer lattice (massive exact ties), and spacings of a few ulp.  Values and first indices must be the oracle's,
    bit for bit."""
    rng = np.random.default_rng(len(case))
    B, N = 2, 1500
    gts = clouds(B, N, 17, "gauss")
    preds = jitter(gts, 3)
    if case == "dups across batches":
        src = rng.integers(0, N, 400)
        dst = rng.integers(0, N, 400)
        gts[0, dst] = gts[0, src]
        preds[1, dst] = preds[1, src]
        preds[0, :200] = gts[0, :200]  # exact coincidences between the clouds too
    elif case == "far from origin":
        gts = (gts * 0.05 + np.asarray((300.0, -200.0, 150.0), np.float32)).astype(np.float32)
        preds = (preds * 0.05 + np.asarray((300.0, -200.0, 150.0), np.float32)).astype(np.float32)
    elif case == "all equal":
        gts[:] = gts[:, :1]
        preds[:] = gts[:, :1]
        preds[1, 700] += 1e-3
    elif case == "lattice":
        gts = rng.integers(-3, 4, size=(B, N, 3)).astype(np.float32)
        preds = rng.integers(-3, 4, size=(B, N, 3)).astype(np.float32)
    else:
        preds = (gts + rng.integers(-2, 3, size=gts.shape) * np.spacing(np.abs(gts))).astype(np.float32)
    for T, RB in ((0, 0), (16, 64), (8, 32)):
        F.tune_nn_bidir(T, RB)
        try:
            m1, a1, m2, a2 = F.nn_bidir(gpu(gts), gpu(preds))
        finally:
            F.tune_nn_bidir(0, 0)
        o1, oa1, o2, oa2 = oracle.nn_bidir(gts, preds, threads=2)
        assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2), (case, T, RB)
        assert np.array_equal(m1.cpu().numpy(), o1) and np.array_equal(m2.cpu().numpy(), o2), (case, T, RB)


def test_nn_bidir_large_cloud_vs_oracle(oracle, F):
    """One configuration-5-sized cloud pair (16384 points, T = 16, RB = 512, four warps per CTA)."""
    gts = clouds(2, 16384, 5)
    preds = jitter(gts, 6)
    preds[1, :3000] = gts[1, 5000:8000]
    m1, a1, m2, a2 = F.nn_bidir(gpu(gts), gpu(preds))
    o1, oa1, o2, oa2 = oracle.nn_bidir(gts, preds, threads=2)
    assert np.array_equal(a1.cpu().numpy(), oa1) and np.array_equal(a2.cpu().numpy(), oa2)
    assert np.array_equal(m1.cpu().numpy(), o1) and np.array_equal(m2.cpu().numpy(), o2)
