"""Argument checks of the feature kNN and edge-feature entry points for clouds past 12800 points.  Every call here is
refused before anything reaches a device (the pointers are never dereferenced), so the test runs without a GPU."""
import hitgeom

HG_E_BADARG, HG_E_UNSUPPORTED = -1, -3
FAKE = 1 << 20  # a 16-byte-aligned address that is never dereferenced: every call below fails its checks first
BIG = 1 << 40   # workspace bytes, past any size check


def _knn(L, B, K, C, k1):
    return L.hg_knn_self_temporal_order_f32(FAKE, B, K, C, k1, None, FAKE, None, 0, None, FAKE, BIG, None)


def test_fp32_knob_past_12800_points_names_the_knob():
    L = hitgeom.lib()
    assert L.hg_tune(b"knn_tc", 1) == 0
    try:
        assert _knn(L, 8, 12801, 64, 20) == HG_E_UNSUPPORTED
        assert b"knn_tc" in L.hg_last_error()
        assert _knn(L, 8, 16384, 128, 40) == HG_E_UNSUPPORTED
        assert b"knn_tc" in L.hg_last_error()
    finally:
        assert L.hg_tune(b"knn_tc", 0) == 0


def test_feature_knn_shapes_past_12800_points_that_no_kernel_takes():
    L = hitgeom.lib()
    for C in (5, 16, 130, 160):  # no multiple of 32 up to 128: the tensor-core kernel does not take them
        assert _knn(L, 1, 12801, C, 20) == HG_E_UNSUPPORTED
    assert _knn(L, 1, 16385, 64, 20) == HG_E_UNSUPPORTED  # past the tensor-core kernel's 16384 points
    assert _knn(L, 1, 16384, 64, 65) == HG_E_BADARG
    assert L.hg_knn_self_temporal_order_f32(FAKE + 4, 1, 16384, 64, 20, None, FAKE, None, 0, None, FAKE, BIG,
                                            None) == HG_E_UNSUPPORTED  # TMA needs a 16-byte-aligned cloud


def test_edge_feature_rejects_bad_arguments():
    L = hitgeom.lib()
    f = L.hg_edge_feature_f32
    assert f(None, FAKE, 1, 64, 16384, 20, FAKE, None) == HG_E_BADARG
    assert f(FAKE, None, 1, 64, 16384, 20, FAKE, None) == HG_E_BADARG
    assert f(FAKE, FAKE, 1, 64, 16384, 20, None, None) == HG_E_BADARG
    for B, C, N, k in ((0, 64, 16384, 20), (1, 0, 16384, 20), (1, 64, 0, 20), (1, 64, 16384, 0), (1, 64, -5, 20)):
        assert f(FAKE, FAKE, B, C, N, k, FAKE, None) == HG_E_BADARG
    assert f(FAKE, FAKE, 1, 64, 1 << 26, 32, FAKE, None) == HG_E_UNSUPPORTED  # N * k >= 2^31
    assert b"N*k" in L.hg_last_error()
