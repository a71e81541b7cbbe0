"""The exact kd-tree of the ordering build (prune_order_kernel, hit-adv_b200/csrc/hg_prune.cu) against a float32 numpy
restatement: pad to a power of two, then per level and segment the box by ordered-int min / max, the axis of the
largest extent, the quantisation scale, the keys (quantised coordinate << 14 | point index) and a sort of the segment.
The permutation and the leaf-box quality H the build stores in a fresh ordering state must be the same bits, for both
norm forms (self-kNN and Chamfer); flagged clouds leave their state untouched."""
import numpy as np
import pytest
import torch

from test_gpu_pruned_search import KINDS, make
from util_inputs import clouds, jitter

pytestmark = pytest.mark.gpu

KQ = np.float32(262142.0)  # kQuantMax
PAD = np.uint64(0xFFFFFFFF)


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def F():
    from hitgeom import functional

    return functional


def ordi(a):  # hg_ord: float32 -> order-preserving uint32
    u = a.view(np.uint32)
    return np.where((u >> np.uint32(31)) != 0, ~u, u | np.uint32(0x80000000)).astype(np.uint32)


def unord(u):  # hg_unord
    u = u.astype(np.uint32)
    return np.where((u & np.uint32(0x80000000)) != 0, u ^ np.uint32(0x80000000), ~u).astype(np.uint32).view(np.float32)


def ref_tree(x):
    """x [N,3] float32 -> (permutation [N] int32, H float32) as the build defines them."""
    N = len(x)
    Np = 64
    while Np < N:
        Np *= 2
    ids = np.full(Np, -1, np.int64)
    ids[:N] = np.arange(N)
    s = Np
    with np.errstate(all="ignore"):
        while s > 32:
            A = ids.reshape(Np // s, s)
            real = A >= 0
            pts = x[np.where(real, A, 0)]  # [nseg, s, 3]
            o = ordi(pts)
            lo = unord(np.where(real[..., None], o, np.uint32(0xFFFFFFFF)).min(1))
            ext = (unord(np.where(real[..., None], o, np.uint32(0)).max(1)) - lo).astype(np.float32)
            r = np.arange(len(A))
            ax = np.where(ext[:, 1] > ext[:, 0], 1, 0)
            ax = np.where(ext[:, 2] > ext[r, ax], 2, ax)
            lo_a, ext_a = lo[r, ax], ext[r, ax]
            scale = np.where(ext_a > 0, KQ / ext_a, np.float32(0)).astype(np.float32)
            c = pts[r[:, None], np.arange(s)[None, :], ax[:, None]]
            f = ((c - lo_a[:, None]).astype(np.float32) * scale[:, None]).astype(np.float32)
            q = np.fmin(np.fmax(f, np.float32(0)), KQ).astype(np.uint64)
            key = np.where(real, (q << np.uint64(14)) | np.where(real, A, 0).astype(np.uint64), PAD)
            key = np.sort(key, axis=1)
            ids = np.where(key == PAD, -1, (key & np.uint64(0x3FFF)).astype(np.int64)).reshape(-1)
            s //= 2
    perm = ids[:N].astype(np.int32)
    # H in the kernel's order: lane 0 of warp w sums leaves w, w + 32, ...; thread 0 sums the 32 partials
    nleaf = (N + 31) // 32
    hw = np.zeros(32, np.float32)
    for L in range(nleaf):
        P = x[perm[L * 32: min(N, L * 32 + 32)]]
        lo, hi = P.min(0), P.max(0)
        e = [np.float32(hi[c] - lo[c]) for c in range(3)]
        hw[L % 32] = np.float32(hw[L % 32] + np.float32(np.float32(e[0] + e[1]) + e[2]))
    H = np.float32(0)
    for w in range(32):
        H = np.float32(H + hw[w])
    return perm, H


def state_of(state, B, N):
    perm = state[: B * N * 4].view(torch.int32).reshape(B, N).cpu().numpy()
    off = (B * N * 4 + 255) // 256 * 256
    hdr = state[off: off + B * 16].view(torch.float32).reshape(B, 4).cpu().numpy()
    return perm, hdr


def cloud(kind, B, N, seed):
    if kind == "flat":  # one axis of zero extent in every segment
        x = clouds(B, N, seed)
        x[..., 1] = np.float32(0.5)
        return x
    if kind == "grid":  # ties in the quantised coordinates: the point index orders them
        rng = np.random.default_rng(seed)
        return (rng.integers(0, 6, (B, N, 3)) * 0.125).astype(np.float32)
    return make(kind, B, N, seed)


def check(x, perm, hdr):
    for b in range(len(x)):
        if not np.all(np.isfinite(x[b])):  # flagged: taken by the all-pairs kernels, the state is left as it was
            assert not perm[b].any() and not hdr[b].any()
            continue
        want_perm, want_H = ref_tree(x[b])
        assert np.array_equal(perm[b], want_perm), f"cloud {b}: permutation differs"
        assert np.float32(hdr[b, 0]).view(np.uint32) == want_H.view(np.uint32), f"cloud {b}: H {hdr[b, 0]} != {want_H}"


@pytest.mark.parametrize("N", [8192, 16384, 12345])
@pytest.mark.parametrize("kind", KINDS + ["flat", "grid"])
def test_order_build_exact_tree(F, kind, N):
    B = 3 if kind == "nonfinite" else 2
    x = cloud(kind, B, N, 31 + N)
    y = x.copy() if kind in ("same", "grid", "nonfinite") else jitter(x, 8)
    order = F.order_state(B, N, "cuda")  # zero-filled: the refit rejects it, the build writes the tree
    F.knn_self(gpu(x), 6, order=order)
    check(x, *state_of(order, B, N))
    go, po = F.order_state(B, N, "cuda"), F.order_state(B, N, "cuda")
    F.nn_bidir(gpu(x), gpu(y), go, po)
    check(x, *state_of(go, B, N))
    check(y, *state_of(po, B, N))
