"""Feature-cloud kNN with lists of 33 to 64 neighbours (DGCNN run with k = 40, model/dgcnn_cls.py:7-13).

Lists longer than 32 take their own kernels: `knn_tc_long_kernel` (tcgen05 TF32 filter + exact FP32 evaluation,
hit-adv_b200/csrc/hg_knn_tc.cu) and `knn_select_rows_kernel<true>` (FP32 tile + row select with a 64-value bound,
hg_knn.cu).  Values and indices (lowest index first on ties) must equal `oracle.knn_self` bit for bit, on every path:
`hg_tune("knn_tc", 2)` forces the tensor-core kernel, `5` its single-sweep variant, `1` the FP32 path."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def gpu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(scope="module")
def F():
    from hitgeom import functional

    return functional


def _knob(value):
    from hitgeom._lib import lib

    lib().hg_tune(b"knn_tc", value)


def feature_clouds(B, K, C, kind, seed):
    """gauss; prototypes (a few distinct rows, half of cloud 1 a single one: massive exact ties, every column a hit);
    scaled (per-row scales e^-4 .. e^4: the TF32 error bound is per row); dups (duplicated points)."""
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
    return np.ascontiguousarray(pc)


def _run(F, pc, k1, knob):
    _knob(knob)
    try:
        vals, idx = F.knn_self(gpu(pc), k1)
    finally:
        _knob(0)
    return vals.cpu().numpy(), idx.cpu().numpy()


# C in {32, 64, 96, 128} x k1 in {33, 40, 64} x K in {300, 1024, 2048, 4096} x four input kinds, covered pairwise
TC_CASES = [(32, 300, 33, "gauss"), (64, 1024, 40, "gauss"), (64, 2048, 64, "prototypes"), (96, 4096, 40, "scaled"),
            (128, 2048, 40, "dups"), (128, 1024, 64, "gauss"), (32, 4096, 64, "dups"), (64, 300, 64, "scaled"),
            (96, 1024, 33, "prototypes"), (128, 4096, 33, "prototypes"), (64, 2048, 40, "scaled"),
            (128, 300, 40, "gauss"), (32, 1024, 40, "prototypes"), (96, 2048, 64, "dups")]


@pytest.mark.parametrize("C,K,k1,kind", TC_CASES)
def test_long_lists_tensor_core_and_fp32_paths_vs_oracle(oracle, F, C, K, k1, kind):
    """Every shape here is one the tensor-core kernel takes (C a multiple of 32, 256 <= K <= 4096); two clouds are too
    few to fill the machine, so the knob forces each path in turn."""
    pc = feature_clouds(2, K, C, kind, C * 7 + K + k1)
    ov, oi = oracle.knn_self(pc, k1, threads=oracle.host_threads())
    for knob in (2, 5, 1):
        vals, idx = _run(F, pc, k1, knob)
        assert np.array_equal(idx, oi), (kind, knob, "indices")
        assert np.array_equal(vals, ov), (kind, knob, "values")


@pytest.mark.parametrize("C,K,k1,kind", [(5, 777, 33, "gauss"), (16, 600, 64, "prototypes"), (130, 1024, 64, "gauss"),
                                         (130, 300, 33, "prototypes"), (16, 2000, 40, "dups"), (5, 70, 64, "gauss"),
                                         (16, 40, 40, "scaled"), (130, 513, 48, "scaled")])
def test_long_lists_generic_channel_counts_vs_oracle(oracle, F, C, K, k1, kind):
    """C no multiple of 32 always takes the FP32 tile + row select.  Prototype clouds put hundreds of exact ties under
    the bound, overflow the 256-entry candidate buffer and take the full-row rounds; K = 70 and 40 leave lanes with
    fewer than two strided elements."""
    pc = feature_clouds(2, K, C, kind, C * 7 + K + k1)
    ov, oi = oracle.knn_self(pc, k1, threads=oracle.host_threads())
    vals, idx = F.knn_self(gpu(pc), k1)
    assert np.array_equal(idx.cpu().numpy(), oi), (kind, "indices")
    assert np.array_equal(vals.cpu().numpy(), ov), (kind, "values")


SAMPLE = [0, 9, 22, 31]  # clouds checked against the oracle in the 32-cloud batches


@pytest.mark.parametrize("C", [64, 128])
def test_long_lists_natural_dispatch_dgcnn_shape(oracle, F, C):
    """32 x 2048 feature clouds at k = 40 with no knob: the default dispatch, the FP32 path and the oracle agree."""
    pc = feature_clouds(32, 2048, C, "gauss", 40 + C)
    vals, idx = F.knn_self(gpu(pc), 40)
    v1, i1 = _run(F, pc, 40, 1)
    vals, idx = vals.cpu().numpy(), idx.cpu().numpy()
    assert np.array_equal(idx, i1) and np.array_equal(vals, v1)
    ov, oi = oracle.knn_self(pc[SAMPLE], 40, threads=oracle.host_threads())
    assert np.array_equal(idx[SAMPLE], oi) and np.array_equal(vals[SAMPLE], ov)


class SmallDGCNN(torch.nn.Module):
    """DGCNN's four EdgeConv layers with the reference's widths (dgcnn_cls.py: 6 -> 64, 128 -> 64, 128 -> 128,
    256 -> 256; 1x1 convolution, LeakyReLU(0.2), max over the k neighbours), built on model_seams' drop-ins.  Records
    every layer's input and kNN graph."""

    def __init__(self, k):
        super().__init__()
        self.k = k
        g = torch.Generator().manual_seed(0)
        self.convs = torch.nn.ModuleList()
        for cin, cout in ((6, 64), (128, 64), (128, 128), (256, 256)):
            conv = torch.nn.Conv2d(cin, cout, kernel_size=1, bias=False)
            with torch.no_grad():
                conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / cin**0.5)
            self.convs.append(conv)
        self.record = []

    def forward(self, x):
        from hitgeom import model_seams

        self.record = []
        feats = []
        for conv in self.convs:
            idx = model_seams.knn(x, self.k)
            self.record.append((x.detach().transpose(2, 1).contiguous().cpu().numpy(), idx.cpu().numpy()))
            e = model_seams.get_graph_feature(x, k=self.k, idx=idx)
            x = torch.nn.functional.leaky_relu(conv(e), 0.2).max(dim=-1)[0]
            feats.append(x)
        return torch.cat(feats, dim=1)


def test_dgcnn_k40_forward_graphs_and_deterministic_backward(oracle):
    """A DGCNN victim with k = 40 at 32 x 2048: every layer's kNN graph (C = 3, 64, 64, 128) is the oracle's on that
    layer's own input, and the backward of a scalar loss gives the same bits twice."""
    rng = np.random.default_rng(40)
    pts = rng.standard_normal((32, 3, 2048)).astype(np.float32)
    pts /= np.abs(pts).max()
    old = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        model = SmallDGCNN(40).cuda()
        grads = []
        for rep in range(2):
            model.zero_grad(set_to_none=True)
            x = gpu(pts).requires_grad_()
            out = model(x)
            if rep == 0:
                assert [r[0].shape[2] for r in model.record] == [3, 64, 64, 128]
                for layer, (inp, idx) in enumerate(model.record):
                    _, oi = oracle.knn_self(inp[SAMPLE], 40, threads=oracle.host_threads())
                    assert np.array_equal(idx[SAMPLE], oi.astype(np.int64)), layer
            (out * out).mean().backward()
            grads.append([x.grad.clone()] + [c.weight.grad.clone() for c in model.convs])
    finally:
        torch.backends.cudnn.deterministic = old
    assert grads[0][0].abs().max() > 0
    for a, b in zip(*grads):
        assert torch.equal(a, b)


@pytest.mark.parametrize("C", [3, 16, 64])
def test_lists_longer_than_64_are_rejected(F, C):
    from hitgeom import HitgeomError, model_seams

    pc = feature_clouds(1, 300, C, "gauss", 1)
    with pytest.raises(HitgeomError):
        F.knn_self(gpu(pc), 65)
    with pytest.raises(HitgeomError):
        model_seams.knn(gpu(pc).transpose(2, 1), 65)
    assert F.knn_self(gpu(pc), 64)[1].shape == (1, 300, 64)
