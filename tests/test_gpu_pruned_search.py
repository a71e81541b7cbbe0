"""The spatially pruned Chamfer / self-kNN passes for large clouds (hit-adv_b200/csrc/hg_prune.cu) against the
all-pairs kernels (switched with hg_tune("prune", 0)) bit for bit, and against the CPU oracle on smaller clouds
forced through the pruned path (hg_tune("prune_min_n", n))."""
import contextlib

import numpy as np
import pytest
import torch

from util_inputs import clouds, jitter

pytestmark = pytest.mark.gpu


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def F():
    from hitgeom import functional

    return functional


@contextlib.contextmanager
def tune(**kv):
    from hitgeom._lib import lib

    for k, v in kv.items():
        assert lib().hg_tune(k.encode(), int(v)) == 0
    try:
        yield
    finally:
        lib().hg_tune(b"prune", 1)
        lib().hg_tune(b"prune_min_n", 0)


def make(kind, B, N, seed):
    rng = np.random.default_rng(seed)
    if kind in ("gauss", "surface"):
        return clouds(B, N, seed, kind)
    if kind == "uniform":
        return rng.uniform(-1, 1, (B, N, 3)).astype(np.float32)
    if kind == "sphere":
        x = rng.standard_normal((B, N, 3))
        return (x / np.linalg.norm(x, axis=-1, keepdims=True)).astype(np.float32)
    if kind == "dups":  # a quarter of the points exactly duplicated elsewhere in the cloud: ties across leaves
        x = clouds(B, N, seed)
        for b in range(B):
            src, dst = rng.permutation(N)[: N // 4], rng.permutation(N)[: N // 4]
            x[b, dst] = x[b, src]
        return x
    if kind == "far":  # norms 1e4, spacings 1e-2: the culling slack is what keeps this exact
        x = 1e4 + 1e-2 * rng.integers(0, 100, (B, N, 3)).astype(np.float32)
        return x.astype(np.float32)
    if kind == "same":  # nothing can be culled
        return np.full((B, N, 3), 0.25, np.float32)
    if kind == "nonfinite":
        x = clouds(B, N, seed)
        x[0, 5, 1] = np.nan
        if B > 1:
            x[1, 7, 0] = np.inf
        return x
    raise ValueError(kind)


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def nn_both(F, gts, preds):
    with tune(prune=0):
        ref = [t.cpu().numpy() for t in F.nn_bidir(gpu(gts), gpu(preds))]
    out = [t.cpu().numpy() for t in F.nn_bidir(gpu(gts), gpu(preds))]
    return ref, out


def knn_both(F, pc, k1):
    with tune(prune=0):
        ref = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1)]
    out = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1)]
    return ref, out


KINDS = ["gauss", "surface", "uniform", "sphere", "dups", "far", "same", "nonfinite"]


@pytest.mark.parametrize("N", [8192, 16384])
@pytest.mark.parametrize("kind", KINDS)
def test_chamfer_pruned_matches_all_pairs(F, kind, N):
    ori = make(kind, 3, N, 11 + N)
    adv = jitter(ori, 5) if kind not in ("same", "nonfinite") else ori.copy()
    ref, out = nn_both(F, ori, adv)
    for r, o in zip(ref, out):
        assert same_bits(r, o)


def test_chamfer_pruned_unequal_sizes(F):
    ori, adv = make("gauss", 2, 16384, 3), jitter(make("gauss", 2, 9000, 4), 6)
    ref, out = nn_both(F, ori, adv)
    for r, o in zip(ref, out):
        assert same_bits(r, o)
    ref, out = nn_both(F, adv, ori)
    for r, o in zip(ref, out):
        assert same_bits(r, o)


@pytest.mark.parametrize("k1", [6, 20, 33])
@pytest.mark.parametrize("N", [8192, 16384])
@pytest.mark.parametrize("kind", KINDS)
def test_knn_pruned_matches_all_pairs(F, kind, N, k1):
    pc = make(kind, 2, N, 21 + N)
    if kind in ("gauss", "surface"):
        pc = jitter(pc, 9)
    ref, out = knn_both(F, pc, k1)
    assert same_bits(ref[0], out[0])
    assert same_bits(ref[1], out[1])


# (non-finite clouds are left out: the oracle propagates NaN like torch, the kernels skip NaN distances, INTEGRATION.md
# section 3; that they keep doing so under the pruned path is checked against the all-pairs kernels above)
@pytest.mark.parametrize("N,kind", [(2048, "gauss"), (3000, "dups"), (4096, "surface"), (2048, "far"),
                                    (2048, "sphere"), (2048, "same")])
def test_pruned_vs_oracle(oracle, F, N, kind):
    ori = make(kind, 2, N, 31 + N)
    adv = jitter(ori, 7) if kind not in ("same", "nonfinite") else ori.copy()
    with tune(prune_min_n=64):
        got = [t.cpu().numpy() for t in F.nn_bidir(gpu(ori), gpu(adv))]
        ref = oracle.nn_bidir(ori, adv, threads=4)
        for r, o in zip(ref, got):
            assert np.array_equal(np.asarray(r), o, equal_nan=True)
        for k1 in (6, 20):
            v, i = F.knn_self(gpu(adv), k1)
            ov, oi = oracle.knn_self(adv, k1, threads=4)
            assert np.array_equal(v.cpu().numpy(), ov, equal_nan=True)
            assert np.array_equal(i.cpu().numpy(), oi)


def test_pruned_knn_temporal_seeds(F):
    pc = jitter(make("gauss", 2, 8192, 41), 3)
    moved = jitter(pc, 8, sigma=0.002, clip=0.01)
    k1 = 6
    stateless = [t.cpu().numpy() for t in F.knn_self(gpu(moved), k1)]
    state = torch.empty((2, 8192, k1), dtype=torch.int32, device="cuda")
    F.knn_self(gpu(pc), k1, state=state, state_valid=False)
    seeded = [t.cpu().numpy() for t in F.knn_self(gpu(moved), k1, state=state, state_valid=True)]
    assert same_bits(stateless[0], seeded[0])
    assert same_bits(stateless[1], seeded[1])
    assert np.array_equal(state.cpu().numpy(), seeded[1])


def test_chamfer_knn_gradient_same_bits(F):
    from hitgeom.dist_utils import ChamferkNNDist

    ori = make("gauss", 2, 8192, 51)
    adv = jitter(ori, 2)

    def grad():
        a = gpu(adv).requires_grad_(True)
        loss = ChamferkNNDist()(a, gpu(ori))
        loss.backward()
        return loss.detach().cpu().numpy(), a.grad.cpu().numpy()

    with tune(prune=0):
        l0, g0 = grad()
    l1, g1 = grad()
    assert same_bits(l0, l1)
    assert same_bits(g0, g1)


@pytest.mark.parametrize("kind", ["gauss", "far", "dups"])
def test_chamfer_p_symmetric(F, kind):
    # P(x_i, y_j) of a pruned pass that puts y in the query role equals the reference's P with x in the row role:
    # nn_bidir(gts=a, preds=b) and nn_bidir(gts=b, preds=a) return each other's (min, arg) pairs bit for bit
    a = make(kind, 2, 8192, 61)
    b = jitter(a, 4) if kind != "far" else make(kind, 2, 8192, 62)
    with tune(prune=0):
        m1, a1, m2, a2 = [t.cpu().numpy() for t in F.nn_bidir(gpu(a), gpu(b))]
        n1, b1, n2, b2 = [t.cpu().numpy() for t in F.nn_bidir(gpu(b), gpu(a))]
    assert same_bits(m1, n2) and same_bits(a1, b2)
    assert same_bits(m2, n1) and same_bits(a2, b1)


@pytest.mark.parametrize("N", [1024, 8192])
def test_knn_seeds_ignore_nan_candidates(F, N):
    # Many NaN points, so that every query's seed scan meets some: a NaN distance must count as +inf in the threshold
    # seeds (grid, Z-order and temporal), or a seed can fall under the true k-th distance and drop real neighbours.
    # Reference: the same all-pairs kernel with cold thresholds (no seeds at all).
    from hitgeom._lib import lib

    pc = make("gauss", 2, N, 71)
    pc[:, ::16, 1] = np.nan
    pc[1, 3::64, 0] = np.inf
    k1 = 6
    try:
        lib().hg_knn_tune_small(-1)
        lib().hg_knn_tune(1 << 30, 0)
        with tune(prune=0):
            cold = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1)]
    finally:
        lib().hg_knn_tune_small(0)
        lib().hg_knn_tune(0, 0)
    with tune(prune=0):
        seeded = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1)]
        state = torch.empty((2, N, k1), dtype=torch.int32, device="cuda")
        F.knn_self(gpu(pc), k1, state=state)
        temporal = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1, state=state, state_valid=True)]
    default = [t.cpu().numpy() for t in F.knn_self(gpu(pc), k1)]
    for other in (seeded, temporal, default):
        assert same_bits(cold[0], other[0])
        assert same_bits(cold[1], other[1])
