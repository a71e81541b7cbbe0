"""DGCNN on clouds of more than 4096 points (model/dgcnn_cls.py at 16384 points per cloud).

Feature kNN beyond 4096 points runs `knn_tc_fused_kernel` / `knn_tc_long_kernel` with per-tile column norms
(hit-adv_b200/csrc/hg_knn_tc.cu); past 12800 points it is the only route.  Edge features beyond 12800 points stage
two planes per pass, one beyond 25600 and none beyond 51200 (hg_edge.cu).  Values and indices must equal
`oracle.knn_self` bit for bit (lowest index first on ties), edge features must equal the torch composition bit for bit,
and a four-layer edge-conv network at 2 x 16384 points must give the logits and input gradient of the same network run
on oracle indices and the torch composition.  Where the reference's Python tree is staged (oracle/_ref/pytree, see
tests/test_gpu_unmodified_callers.py), its own DGCNN runs the same comparison."""
import os
import subprocess
import sys
import tempfile
import textwrap
import types

import numpy as np
import pytest
import torch

from util_inputs import normwise

pytestmark = pytest.mark.gpu


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _knob(value):
    from hitgeom._lib import lib

    assert lib().hg_tune(b"knn_tc", value) == 0


def feature_clouds(B, K, C, kind, seed):
    """gauss; prototypes (five distinct rows, half of cloud 1 a single one: massive exact ties, every column a hit);
    scaled (per-row scales e^-4 .. e^4: the TF32 error bound is per row); dups (duplicated points, among them pairs on
    both sides of every 256-column tile boundary past 4096, and copies of one early row there)."""
    rng = np.random.default_rng(seed)
    pc = rng.standard_normal((B, K, C)).astype(np.float32)
    if kind == "prototypes":
        protos = rng.standard_normal((5, C)).astype(np.float32)
        pc = protos[rng.integers(0, 5, size=(B, K))]
        pc[min(1, B - 1), : K // 2] = protos[0]
    elif kind == "scaled":
        pc *= np.exp(rng.uniform(-4, 4, size=(B, K, 1))).astype(np.float32)
    elif kind == "dups":
        pc[0, K // 10 : K // 3] = pc[0, K // 2 : K // 2 + (K // 3 - K // 10)]
        pc[-1, :] = pc[-1, rng.integers(0, 64, size=K)]
        for t in range(4096, K, 256):
            pc[0, t - 1] = pc[0, t] = pc[0, 5]
    return np.ascontiguousarray(pc)


def _run(F, pc, k1, knob):
    _knob(knob)
    try:
        vals, idx = F.knn_self(gpu(pc), k1)
    finally:
        _knob(0)
    return vals.cpu().numpy(), idx.cpu().numpy()


# C in {32, 64, 96, 128} x k1 in {1, 20, 32, 33, 40, 64} x K in {4097, 8192, 12801, 16384} x four input kinds, covered
# pairwise
TC_CASES = [(32, 4097, 1, "gauss"), (32, 16384, 20, "prototypes"), (32, 12801, 32, "scaled"), (32, 8192, 33, "dups"),
            (32, 16384, 40, "gauss"), (32, 12801, 64, "prototypes"), (64, 8192, 1, "prototypes"),
            (64, 4097, 20, "scaled"), (64, 16384, 32, "dups"), (64, 12801, 33, "gauss"), (64, 4097, 40, "prototypes"),
            (64, 16384, 64, "scaled"), (96, 12801, 1, "scaled"), (96, 8192, 20, "dups"), (96, 4097, 32, "gauss"),
            (96, 16384, 33, "prototypes"), (96, 8192, 40, "scaled"), (96, 4097, 64, "dups"), (128, 16384, 1, "dups"),
            (128, 12801, 20, "gauss"), (128, 8192, 32, "prototypes"), (128, 4097, 33, "scaled"),
            (128, 12801, 40, "dups"), (128, 8192, 64, "gauss")]


@pytest.fixture(scope="module")
def F():
    from hitgeom import functional

    return functional


@pytest.mark.parametrize("case", range(len(TC_CASES)))
def test_large_feature_knn_tensor_core_vs_oracle(oracle, F, case):
    """The tensor-core kernel with per-tile norms, two-pass (knob 2) and single-sweep (knob 5), against the oracle;
    one or two clouds."""
    C, K, k1, kind = TC_CASES[case]
    B = 2 if case % 2 == 0 else 1
    pc = feature_clouds(B, K, C, kind, C * 7 + K + k1)
    ov, oi = oracle.knn_self(pc, k1, threads=oracle.host_threads())
    for knob in (2, 5):
        vals, idx = _run(F, pc, k1, knob)
        assert np.array_equal(idx, oi), (kind, knob, "indices")
        assert np.array_equal(vals, ov), (kind, knob, "values")


@pytest.mark.parametrize("K,C,k1", [(6000, 64, 20), (8192, 128, 40), (12800, 64, 40), (12800, 128, 20)])
def test_tensor_core_and_fp32_routes_agree_up_to_12800(F, K, C, k1):
    """Between 4097 and 12800 points both routes run: hg_tune("knn_tc", 1) (FP32 tile + row select) and 2 (tensor
    cores) give the same bits, and so does the default dispatch."""
    pc = feature_clouds(2, K, C, "gauss", K + C + k1)
    v1, i1 = _run(F, pc, k1, 1)
    v2, i2 = _run(F, pc, k1, 2)
    v0, i0 = _run(F, pc, k1, 0)
    assert np.array_equal(i1, i2) and np.array_equal(v1, v2)
    assert np.array_equal(i0, i2) and np.array_equal(v0, v2)


def test_fp32_knob_past_12800_points_is_refused(F):
    from hitgeom import HitgeomError

    pc = feature_clouds(1, 12801, 64, "gauss", 3)
    _knob(1)
    try:
        with pytest.raises(HitgeomError, match="knn_tc"):
            F.knn_self(gpu(pc), 20)
    finally:
        _knob(0)
    assert F.knn_self(gpu(pc), 20)[1].shape == (1, 12801, 20)


def _edge_idx(B, N, k, seed):
    """random neighbours, the point itself first (as DGCNN's kNN gives it) and a hub: point 0 receives N/8 extra edges"""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    idx = torch.randint(0, N, (B, N, k), generator=gen, device="cuda")
    idx[:, :, 0] = torch.arange(N, device="cuda")[None, :]
    if k > 1:
        idx[:, : N // 8, 1] = 0
    return idx.contiguous()


@pytest.mark.parametrize("N", [12800, 12801, 16384, 25601, 51201])
@pytest.mark.parametrize("k", [20, 40, 7])
@pytest.mark.parametrize("C", [3, 64])
def test_large_edge_features_vs_torch_program(N, k, C):
    """Four staged planes per pass up to 12800 points, two up to 25600, one up to 51200, none beyond; k % 4 == 0 takes
    the float4 path.  Forward bit-identical to cat(x[idx] - x, x); backward within 1e-5 norm-wise of autograd."""
    from hitgeom import functional as F
    from oracle import torch_port as tp

    B = 2 if N * C <= 16384 * 64 else 1
    gen = torch.Generator(device="cuda").manual_seed(N + k + C)
    x = torch.randn(B, C, N, generator=gen, device="cuda")
    idx = _edge_idx(B, N, k, N * k + C)
    w = torch.randn(B, 2 * C, N, k, generator=gen, device="cuda")
    xr = x.clone().requires_grad_()
    ref = tp.get_graph_feature(xr, idx)
    (ref * w).sum().backward()
    xm = x.clone().requires_grad_()
    out = F.edge_feature(xm, idx)
    assert torch.equal(out, ref)
    del ref
    (out * w).sum().backward()
    assert normwise(xm.grad.cpu().numpy(), xr.grad.cpu().numpy()) < 1e-5


# ---- DGCNN end to end at 2 x 16384 points ----------------------------------------------------------------------------
class EdgeConvNet(torch.nn.Module):
    """DGCNN's four EdgeConv layers with the reference's widths (dgcnn_cls.py: 6 -> 64, 128 -> 64, 128 -> 128,
    256 -> 256; 1x1 convolution, LeakyReLU(0.2), max over the k neighbours), then max-pooling over the points and a
    linear head to 40 logits.  `knn` and `get_graph_feature` are looked up in `seams` at call time, as the reference
    model looks them up in its module's globals."""

    def __init__(self, k, seams):
        super().__init__()
        self.k, self.seams = k, seams
        g = torch.Generator().manual_seed(0)
        self.convs = torch.nn.ModuleList()
        for cin, cout in ((6, 64), (128, 64), (128, 128), (256, 256)):
            conv = torch.nn.Conv2d(cin, cout, kernel_size=1, bias=False)
            with torch.no_grad():
                conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / cin**0.5)
            self.convs.append(conv)
        self.head = torch.nn.Linear(512, 40)
        with torch.no_grad():
            self.head.weight.copy_(torch.randn(self.head.weight.shape, generator=g) / 512**0.5)
            self.head.bias.zero_()

    def forward(self, x):
        feats = []
        for conv in self.convs:
            e = self.seams.get_graph_feature(x, k=self.k)
            x = torch.nn.functional.leaky_relu(conv(e), 0.2).max(dim=-1)[0]
            feats.append(x)
        return self.head(torch.cat(feats, dim=1).max(dim=-1)[0])


def _reference_seams(oracle):
    """A stand-in for model/dgcnn_cls.py's module: knn returns the oracle's indices, get_graph_feature is the torch
    composition of the reference."""
    from oracle import torch_port as tp

    mod = types.ModuleType("model.dgcnn_cls")

    def knn(x, k):
        pc = x.detach().transpose(2, 1).contiguous().cpu().numpy()
        _, oi = oracle.knn_self(pc, k, threads=oracle.host_threads())
        return torch.from_numpy(oi.astype(np.int64)).to(x.device)

    def get_graph_feature(x, k=20, idx=None, dim9=False):
        if idx is None:
            idx = mod.knn(x if not dim9 else x[:, 6:], k=k)
        return tp.get_graph_feature(x, idx)

    mod.knn, mod.get_graph_feature = knn, get_graph_feature
    return mod


@pytest.mark.parametrize("k", [20, 40])
def test_dgcnn_16384_points_through_patch_reference(oracle, k):
    """B = 2 x 16384 points.  The network runs once over the stand-in module (oracle + torch), then again after
    `hitgeom.patch_reference()` has rebound that module's knn and get_graph_feature to hitgeom's seams; logits and the
    input gradient agree to 1e-4 norm-wise."""
    import hitgeom
    from hitgeom import model_seams

    rng = np.random.default_rng(k)
    pts = rng.standard_normal((2, 3, 16384)).astype(np.float32)
    pts /= np.abs(pts).max()
    saved = sys.modules.get("model.dgcnn_cls")
    mod = _reference_seams(oracle)
    sys.modules["model.dgcnn_cls"] = mod
    try:
        model = EdgeConvNet(k, mod).cuda()
        runs = []
        for patched in (False, True):
            if patched:
                assert "model.dgcnn_cls" in hitgeom.patch_reference()
                assert mod.knn is model_seams.knn and mod.get_graph_feature is model_seams.get_graph_feature
            x = gpu(pts).requires_grad_()
            logits = model(x)
            (logits * logits).sum().backward()
            runs.append((logits.detach().cpu().numpy(), x.grad.cpu().numpy()))
    finally:
        if saved is None:
            sys.modules.pop("model.dgcnn_cls", None)
        else:
            sys.modules["model.dgcnn_cls"] = saved
    (l_ref, g_ref), (l_me, g_me) = runs
    assert np.abs(g_ref).max() > 0
    assert normwise(l_me, l_ref) < 1e-4
    assert normwise(g_me, g_ref) < 1e-4


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREE = os.path.join(ROOT, "oracle", "_ref", "pytree")

REF_SCRIPT = textwrap.dedent('''
    import inspect, os, sys, types
    sys.dont_write_bytecode = True
    ROOT, TREE = %(root)r, %(tree)r
    sys.path[:0] = [TREE, os.path.join(TREE, "pointnet2_ops_lib"), os.path.join(ROOT, "hit-adv_b200"), ROOT,
                    os.path.join(ROOT, "tests")]
    import numpy as np, torch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    for name in ("mayavi", "mayavi.mlab", "open3d", "matplotlib", "matplotlib.pyplot", "seaborn", "h5py"):
        sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].use = lambda *a, **k: None
    sys.modules["seaborn"].set = lambda *a, **k: None
    import hitgeom
    from hitgeom import model_seams as ms
    from oracle import oracle as O
    from util_inputs import normwise
    hitgeom.install()
    import model.dgcnn_cls as dg
    assert dg.__file__.startswith(TREE), dg.__file__
    O.build()

    def oracle_knn(x, k):  # the reference's own get_graph_feature calls this through the module's globals
        pc = x.detach().transpose(2, 1).contiguous().cpu().numpy()
        _, oi = O.knn_self(pc, k, threads=O.host_threads())
        return torch.from_numpy(oi.astype(np.int64)).to(x.device)

    K = int(os.environ["DGCNN_K"])
    params = inspect.signature(dg.DGCNN.__init__).parameters
    if "args" in params:
        model = dg.DGCNN(types.SimpleNamespace(k=K, emb_dims=1024, dropout=0.5))
    else:
        model = dg.DGCNN(**{n: v for n, v in (("k", K), ("emb_dims", 1024)) if n in params})
    torch.manual_seed(0)
    model = model.cuda().eval()
    rng = np.random.default_rng(K)
    pts = rng.standard_normal((2, 3, 16384)).astype(np.float32)
    pts /= np.abs(pts).max()
    runs = []
    dg.knn = oracle_knn
    for patched in (False, True):
        if patched:
            assert "model.dgcnn_cls" in hitgeom.patch_reference()
            assert dg.knn is ms.knn and dg.get_graph_feature is ms.get_graph_feature
        x = torch.from_numpy(pts).cuda().requires_grad_()
        out = model(x)
        logits = out[0] if isinstance(out, tuple) else out
        (logits * logits).sum().backward()
        runs.append((logits.detach().cpu().numpy(), x.grad.cpu().numpy()))
    (l_ref, g_ref), (l_me, g_me) = runs
    assert np.abs(g_ref).max() > 0
    assert normwise(l_me, l_ref) < 1e-4, normwise(l_me, l_ref)
    assert normwise(g_me, g_ref) < 1e-4, normwise(g_me, g_ref)
    print("DGCNN_REF_OK", normwise(l_me, l_ref), normwise(g_me, g_ref))
''')


@pytest.mark.skipif(not os.path.isdir(TREE), reason="needs the unmodified TRLou/HiT-ADV Python tree in oracle/_ref/pytree: "
                                                    "HITADV_REFERENCE=<checkout> python oracle/stage_ref.py")
@pytest.mark.parametrize("k", [20, 40])
def test_reference_dgcnn_16384_points_through_patch_reference(k):
    """The reference's own DGCNN (model/dgcnn_cls.py, file unchanged, eval mode) at 2 x 16384 points: once with its
    own get_graph_feature over oracle indices, once after `hitgeom.patch_reference()`; logits and the input gradient
    agree to 1e-4 norm-wise.  In a subprocess: `hitgeom.install()` rewires sys.modules."""
    out = subprocess.run([sys.executable, "-c", REF_SCRIPT % {"root": ROOT, "tree": TREE}], capture_output=True,
                         text=True, timeout=900, cwd=tempfile.gettempdir(), env=dict(os.environ, DGCNN_K=str(k)))
    assert out.returncode == 0 and "DGCNN_REF_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-4000:])
