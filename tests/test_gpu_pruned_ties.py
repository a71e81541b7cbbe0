"""Tie order of the pruned self-kNN search (hit-adv_b200/csrc/hg_prune.cu) in every list size it instantiates.

A list of KM = 6, 20, 32 or 64 entries serves every k + 1 up to KM; with k + 1 < KM only its last k + 1 entries are
live.  On a shuffled lattice most distances are exact and equal many times over, so the lowest original index among
equal values decides almost every list; the result must equal the CPU oracle bit for bit."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def lattice(B, N, seed):
    """B clouds of N points of a 16 x 16 x 8 lattice of spacing 1/16 (exact squared distances), each in its own random
    order, so that equal distances come from leaves all over the tree."""
    g = np.stack(np.meshgrid(np.arange(16), np.arange(16), np.arange(8), indexing="ij"), -1).reshape(-1, 3)
    rng = np.random.default_rng(seed)
    return np.stack([g[rng.permutation(len(g))[:N]] / 16.0 for _ in range(B)]).astype(np.float32)


@pytest.mark.parametrize("k1", [5, 19, 31, 40])  # lists of 6, 20, 32 and 64 entries
def test_pruned_knn_tie_order_vs_oracle(oracle, k1):
    from hitgeom import functional as F
    from hitgeom._lib import lib

    pc = lattice(2, 2000, 81 + k1)  # 2000 points: the last leaf is partly padding
    assert lib().hg_tune(b"prune_min_n", 64) == 0
    try:
        v, i = F.knn_self(torch.from_numpy(pc).cuda(), k1)
    finally:
        lib().hg_tune(b"prune_min_n", 0)
    ov, oi = oracle.knn_self(pc, k1, threads=4)
    assert np.array_equal(v.cpu().numpy().view(np.uint32), ov.view(np.uint32))
    assert np.array_equal(i.cpu().numpy(), oi)
