"""Ordering states of the pruned passes (hg_nn_bidir_temporal_f32, hg_knn_self_temporal_order_f32, the loss classes'
temporal_seeds): a call with a state refits the stored kd-tree permutation instead of rebuilding it, and must return the
same bits as the stateless call whatever the state holds -- first use, a nearby cloud, an unrelated cloud, corrupt
contents."""
import contextlib

import numpy as np
import pytest
import torch

from test_gpu_pruned_search import KINDS, make, same_bits
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
        lib().hg_tune(b"prune_refit_stage", 0)


@contextlib.contextmanager
def counting(F):
    """Yields a function returning the ordering counters (refit and kept, rebuilt from a state, built without one) since
    the previous read."""
    from hitgeom._lib import lib

    assert lib().hg_tune(b"prune_count", 1) == 0
    F.prune_order_counters()
    try:
        yield F.prune_order_counters
    finally:
        lib().hg_tune(b"prune_count", 0)
        F.prune_order_counters()


def perm_of(state, B, N):
    return state[: B * N * 4].view(torch.int32).reshape(B, N).cpu().numpy().copy()


def header_of(state, B, N):
    off = (B * N * 4 + 255) // 256 * 256
    return state[off: off + B * 16].view(torch.float32).reshape(B, 4)


def outs(ts):
    return [t.cpu().numpy() for t in ts]


def assert_same(ref, got):
    for r, o in zip(ref, got):
        assert same_bits(r, o)


def is_perm(p):
    N = p.shape[1]
    return all(np.array_equal(np.sort(row), np.arange(N)) for row in p)


@pytest.mark.parametrize("N", [8192, 16384])
@pytest.mark.parametrize("kind", KINDS)
def test_nn_bidir_state_first_refit_rebuild(F, kind, N):
    B = 3
    ori = make(kind, B, N, 11 + N)
    adv = jitter(ori, 5) if kind not in ("same", "nonfinite") else ori.copy()
    steady = kind in ("same", "nonfinite")  # clouds that cannot move without changing kind
    moved = adv if steady else jitter(adv, 6, sigma=1e-4, clip=5e-4)
    other = make(kind, B, N, 99 + N)
    other_adv = jitter(other, 7) if not steady else other.copy()
    go, po = F.order_state(B, N, "cuda"), F.order_state(B, N, "cuda")
    flagged = kind == "nonfinite"
    refs = [outs(F.nn_bidir(gpu(g), gpu(p))) for g, p in ((ori, adv), (ori, moved), (other, other_adv))]
    with counting(F) as counts:
        # first call: zero-filled states fail validation, every unflagged cloud is built from the state
        assert_same(refs[0], outs(F.nn_bidir(gpu(ori), gpu(adv), go, po)))
        c = counts()
        assert c[2] == 0
        if not flagged:
            assert c == (0, 2 * B, 0)
        p_go, p_po = perm_of(go, B, N), perm_of(po, B, N)
        if not flagged:
            assert is_perm(p_go) and is_perm(p_po)
        # second call, ori unchanged and adv moved a little: both refit and kept, permutations unchanged
        assert_same(refs[1], outs(F.nn_bidir(gpu(ori), gpu(moved), go, po)))
        assert counts() == (2 * B, 0, 0)
        assert np.array_equal(perm_of(go, B, N), p_go) and np.array_equal(perm_of(po, B, N), p_po)
        # an unrelated cloud of the same shape: the stale orderings' boxes are far too large, so they are rebuilt
        assert_same(refs[2], outs(F.nn_bidir(gpu(other), gpu(other_adv), go, po)))
        c = counts()
        if kind not in ("same", "nonfinite"):
            assert c == (0, 2 * B, 0)
            assert not np.array_equal(perm_of(go, B, N), p_go)


@pytest.mark.parametrize("corrupt", ["duplicate", "out_of_range", "negative", "nan_header", "zeros", "random"])
def test_nn_bidir_corrupt_state(F, corrupt):
    B, N = 3, 8192
    ori = make("gauss", B, N, 5)
    adv = jitter(ori, 6)
    go, po = F.order_state(B, N, "cuda"), F.order_state(B, N, "cuda")
    F.nn_bidir(gpu(ori), gpu(adv), go, po)
    for st in (go, po):
        p = st[: B * N * 4].view(torch.int32).reshape(B, N)
        if corrupt == "duplicate":
            p[:, 1] = p[:, 0]
        elif corrupt == "out_of_range":
            p[1, 77] = N
        elif corrupt == "negative":
            p[2, 5] = -3
        elif corrupt == "nan_header":
            header_of(st, B, N)[:, 0] = float("nan")
        elif corrupt == "zeros":
            st.zero_()
        else:
            st.copy_(torch.randint(0, 256, st.shape, dtype=torch.uint8, generator=torch.Generator().manual_seed(3)))
    ref = outs(F.nn_bidir(gpu(ori), gpu(adv)))
    with counting(F) as counts:
        assert_same(ref, outs(F.nn_bidir(gpu(ori), gpu(adv), go, po)))
        c = counts()
    if corrupt in ("duplicate", "nan_header", "zeros", "random"):
        assert c == (0, 2 * B, 0)
    else:  # one cloud of each state corrupted
        assert c == (2 * (B - 1), 2, 0)
    assert is_perm(perm_of(go, B, N)) and is_perm(perm_of(po, B, N))
    assert np.isfinite(header_of(go, B, N).cpu().numpy()[:, 0]).all()


@pytest.mark.parametrize("stage", [1, 2])
def test_refit_gather_modes(F, stage):
    # the refit's gather from the cloud staged in shared memory (1) or from global memory (2): same orderings
    B, N = 2, 16384
    ori, adv = make("dups", B, N, 8), jitter(make("dups", B, N, 8), 9)
    moved = jitter(adv, 10, sigma=1e-4, clip=5e-4)
    ref = outs(F.nn_bidir(gpu(ori), gpu(moved)))
    go, po = F.order_state(B, N, "cuda"), F.order_state(B, N, "cuda")
    with tune(prune_refit_stage=stage):
        F.nn_bidir(gpu(ori), gpu(adv), go, po)
        with counting(F) as counts:
            assert_same(ref, outs(F.nn_bidir(gpu(ori), gpu(moved), go, po)))
            assert counts() == (2 * B, 0, 0)


def test_nn_bidir_state_unequal_sizes_and_one_state(F):
    B = 2
    ori, adv = make("gauss", B, 16384, 3), jitter(make("gauss", B, 9000, 4), 6)
    for gts, preds in ((ori, adv), (adv, ori)):
        N2, N1 = gts.shape[1], preds.shape[1]
        ref = outs(F.nn_bidir(gpu(gts), gpu(preds)))
        go, po = F.order_state(B, N2, "cuda"), F.order_state(B, N1, "cuda")
        for _ in range(2):
            assert_same(ref, outs(F.nn_bidir(gpu(gts), gpu(preds), go, po)))
            assert_same(ref, outs(F.nn_bidir(gpu(gts), gpu(preds), gts_order=go)))
            assert_same(ref, outs(F.nn_bidir(gpu(gts), gpu(preds), preds_order=po)))
    with pytest.raises(RuntimeError):  # a state too small for its cloud
        F.nn_bidir(gpu(ori), gpu(adv), gts_order=F.order_state(B, 9000, "cuda"))
    st = F.order_state(B, 16384, "cuda")
    with pytest.raises(RuntimeError):  # one buffer for both clouds
        F.nn_bidir(gpu(ori), gpu(ori), st, st)


@pytest.mark.parametrize("valid", [False, True])
@pytest.mark.parametrize("k1", [6, 20, 33])
@pytest.mark.parametrize("N", [8192, 16384])
def test_knn_order_state(F, N, k1, valid):
    B = 2
    pc = jitter(make("gauss", B, N, 41), 3)
    moved = jitter(pc, 8, sigma=1e-4, clip=5e-4)
    ref0, ref = outs(F.knn_self(gpu(pc), k1)), outs(F.knn_self(gpu(moved), k1))
    order = F.order_state(B, N, "cuda")
    state = torch.empty((B, N, k1), dtype=torch.int32, device="cuda")
    with counting(F) as counts:
        assert_same(ref0, outs(F.knn_self(gpu(pc), k1, state=state, order=order)))
        assert counts() == (0, B, 0)
        p0 = perm_of(order, B, N)
        got = outs(F.knn_self(gpu(moved), k1, state=state, state_valid=valid, order=order))
        assert counts() == (B, 0, 0)
    assert_same(ref, got)
    assert np.array_equal(perm_of(order, B, N), p0)
    assert np.array_equal(state.cpu().numpy(), got[1])


@pytest.mark.parametrize("k1", [33, 64])
def test_pruned_temporal_seeds_long_lists(F, k1):
    # lists longer than the 32 previous neighbours the temporal seed kernel bounds: no seeds, same results
    B, N = 2, 8192
    pc = jitter(make("gauss", B, N, 43), 3)
    moved = jitter(pc, 8, sigma=1e-4, clip=5e-4)
    state = torch.empty((B, N, k1), dtype=torch.int32, device="cuda")
    F.knn_self(gpu(pc), k1, state=state)
    assert_same(outs(F.knn_self(gpu(moved), k1)), outs(F.knn_self(gpu(moved), k1, state=state, state_valid=True)))


@pytest.mark.parametrize("kind", KINDS)
def test_knn_order_state_kinds(F, kind):
    B, N, k1 = 2, 8192, 6
    pc = make(kind, B, N, 21 + N)
    if kind in ("gauss", "surface"):
        pc = jitter(pc, 9)
    order = F.order_state(B, N, "cuda")
    for cloud in (pc, make(kind, B, N, 5), pc):
        assert_same(outs(F.knn_self(gpu(cloud), k1)), outs(F.knn_self(gpu(cloud), k1, order=order)))


def test_order_state_shared_between_chamfer_and_knn(F):
    # one state for the Chamfer call (Chamfer norm arithmetic) and the kNN call (KNNDist's) on the same cloud
    B, N = 2, 16384
    ori, adv = make("surface", B, N, 1), jitter(make("surface", B, N, 1), 2)
    go, po = F.order_state(B, N, "cuda"), F.order_state(B, N, "cuda")
    with counting(F) as counts:
        for _ in range(2):
            assert_same(outs(F.nn_bidir(gpu(ori), gpu(adv))), outs(F.nn_bidir(gpu(ori), gpu(adv), go, po)))
            assert_same(outs(F.knn_self(gpu(adv), 6)), outs(F.knn_self(gpu(adv), 6, order=po)))
        # with states: 2 rebuilds (first Chamfer call), then 4 refits; stateless: 2 + 1 builds per round
        assert counts() == (4 * B, 2 * B, 6 * B)


@pytest.mark.parametrize("N,kind", [(2048, "gauss"), (3000, "dups"), (2048, "far")])
def test_order_state_vs_oracle(oracle, F, N, kind):
    ori = make(kind, 2, N, 31 + N)
    adv = jitter(ori, 7)
    with tune(prune_min_n=64):
        go, po, ko = (F.order_state(2, N, "cuda") for _ in range(3))
        for step in range(2):
            a = adv if step == 0 else jitter(adv, 8, sigma=1e-4, clip=5e-4)
            got = outs(F.nn_bidir(gpu(ori), gpu(a), go, po))
            for r, o in zip(oracle.nn_bidir(ori, a, threads=4), got):
                assert np.array_equal(np.asarray(r), o, equal_nan=True)
            v, i = F.knn_self(gpu(a), 6, order=ko)
            ov, oi = oracle.knn_self(a, 6, threads=4)
            assert np.array_equal(v.cpu().numpy(), ov, equal_nan=True)
            assert np.array_equal(i.cpu().numpy(), oi)


def _trajectory(B, N, steps, lr, seed):
    rng = np.random.default_rng(seed)
    ori = clouds(B, N, seed)
    adv = ori.copy()
    out = []
    for _ in range(steps):
        adv = np.clip(adv + lr * np.sign(rng.standard_normal(adv.shape)), ori - 0.05, ori + 0.05).astype(np.float32)
        out.append(adv.copy())
    return ori, out


@pytest.mark.parametrize("name", ["ChamferDist", "HausdorffDist", "KNNDist", "ChamferkNNDist"])
def test_loss_classes_temporal_same_bits(F, name):
    from hitgeom import dist_utils

    cls = getattr(dist_utils, name)
    B, N = 2, 8192
    ori, traj = _trajectory(B, N, 5, 5e-4, 17)
    mod = cls().temporal_seeds(True)
    ori_d = gpu(ori)

    def run(m, adv):
        a = gpu(adv).requires_grad_(True)
        loss = m(a) if name == "KNNDist" else m(a, ori_d)
        loss.backward()
        return loss.detach().cpu().numpy(), a.grad.cpu().numpy()

    with counting(F) as counts:
        for t, adv in enumerate(traj):
            l1, g1 = run(mod, adv)
            c = counts()
            l0, g0 = run(cls(), adv)
            counts()
            assert same_bits(l0, l1) and same_bits(g0, g1), (name, t)
            if t >= 1:  # steady state: every ordering of the step refit and kept
                n = {"KNNDist": 1, "ChamferkNNDist": 3}.get(name, 2)
                assert c == (n * B, 0, 0), (name, t, c)


def test_channel_first_chamfer_takes_no_state(F):
    # HiT-ADV's degenerate [B,3,K] call (generic-D path): no state is kept
    from hitgeom.dist_utils import ChamferDist

    x = gpu(clouds(2, 64, 3)).transpose(1, 2).contiguous()
    y = gpu(clouds(2, 64, 4)).transpose(1, 2).contiguous()
    m = ChamferDist().temporal_seeds(True)
    assert same_bits(m(x, y).cpu().numpy(), ChamferDist()(x, y).cpu().numpy())
    assert m._orders == {}


def test_graph_replay_with_order_states_is_bit_identical():
    """CW-kNN on clouds forced onto the pruned path: eager without states, eager with them (CWKNN switches
    temporal_seeds on), and the captured iteration replayed -- the same adversarial clouds bit for bit."""
    from hitgeom.adv_utils import UntargetedLogitsAdvLoss
    from hitgeom.cw_knn import CWUKNN
    from hitgeom.dist_utils import ChamferkNNDist
    from util_models import TinyPointNet

    class Stateless(torch.nn.Module):  # no temporal_seeds method: CWKNN keeps it stateless
        def __init__(self):
            super().__init__()
            self.d = ChamferkNNDist()

        def forward(self, a, o):
            return self.d(a, o)

    pts = torch.from_numpy(clouds(8, 1024, 77))
    res = []
    with tune(prune_min_n=1024):
        for dist, graph in ((Stateless(), False), (ChamferkNNDist(), False), (ChamferkNNDist(), True)):
            model = TinyPointNet(40, seed=1)
            with torch.no_grad():
                label = model(pts.transpose(1, 2)).argmax(1)
            atk = CWUKNN(model, UntargetedLogitsAdvLoss(kappa=10.), dist, None, attack_lr=1e-2, num_iter=20,
                         graph=graph, capturable_adam=True)
            torch.manual_seed(3)
            res.append(atk.attack(pts, label))
    for adv, succ in res[1:]:
        np.testing.assert_array_equal(res[0][0], adv)
        assert succ == res[0][1]


SENTINEL = 0xAB


def _sentinel(nbytes):
    return torch.full((nbytes,), SENTINEL, dtype=torch.uint8, device="cuda")


@pytest.mark.parametrize("case", ["D4", "small_N", "prune_off"])
def test_state_untouched_when_path_does_not_apply(F, case):
    B = 2
    N, D = (1024, 3) if case == "small_N" else (8192, 4 if case == "D4" else 3)
    rng = np.random.default_rng(1)
    a = rng.standard_normal((B, N, D)).astype(np.float32)
    b = rng.standard_normal((B, N, D)).astype(np.float32)
    nbytes = F.order_state(B, N, "cuda").numel()
    go, po, ko = _sentinel(nbytes), _sentinel(nbytes), _sentinel(nbytes)
    with tune(prune=0 if case == "prune_off" else 1):
        ref = outs(F.nn_bidir(gpu(a), gpu(b)))
        assert_same(ref, outs(F.nn_bidir(gpu(a), gpu(b), go, po)))
        if D == 3:
            assert_same(outs(F.knn_self(gpu(a), 6)), outs(F.knn_self(gpu(a), 6, order=ko)))
    torch.cuda.synchronize()
    for st in (go, po, ko):
        assert bool((st == SENTINEL).all())
