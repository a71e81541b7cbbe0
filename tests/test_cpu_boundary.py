"""CPU-side checks of the drop-in boundary: the C-ABI library builds for sm_100a, loads, and exports every
symbol that include/hitgeom.h declares; the product package never touches the oracle; the mirror classes
keep the reference's names and signatures; everything fails loudly without a CUDA device."""
import inspect
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "hit-adv_b200")


def header_symbols():
    src = open(os.path.join(ROOT, "include", "hitgeom.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    import hitgeom

    L = hitgeom.lib()  # raises if libhitgeom.so is missing or a bound symbol is absent
    syms = header_symbols()
    assert len(syms) >= 30
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/hitgeom.h but not exported"
    assert L.hg_version() >= 100
    bound = set(hitgeom.exported_symbols())
    missing = [s for s in syms if s not in bound]
    assert not missing, f"declared but not bound in _lib.py: {missing}"


def test_library_contains_only_sm100a_code():
    so = os.path.join(PKG, "hitgeom", "libhitgeom.so")
    out = subprocess.run(["cuobjdump", "-lelf", so], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_packed_fp32_and_warp_reduce_instructions_present():
    """The hot kernel is built from Blackwell's packed FP32 pipe ops and the f32 warp-reduce (sm_100a)."""
    so = os.path.join(PKG, "hitgeom", "libhitgeom.so")
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    for mnemonic in ("FFMA2", "FADD2", "FMUL2", "FMNMX3", "CREDUX.MIN.F32"):
        assert mnemonic in sass, mnemonic


def test_tune_keys():
    """hg_tune accepts the knobs the suite sets and refuses removed ones (it only sets host flags: no device needed)."""
    import hitgeom

    L = hitgeom.lib()
    for key in (b"nn_exact", b"fps_threads", b"scatter", b"knn_win"):
        assert L.hg_tune(key, 0) != 0, key
        assert key in L.hg_last_error()
    defaults = {b"knn_tc": 0, b"small_fused": 0, b"prune": 1, b"prune_min_n": 0, b"prune_count": 0,
                b"prune_refit_stage": 0}
    for key, value in defaults.items():
        assert L.hg_tune(key, value) == 0, key


def test_product_never_imports_the_oracle():
    bad = []
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="replace").read()
                if re.search(r"\boracle\b", txt) and "liboracle" in txt or re.search(r"(import|from)\s+oracle", txt):
                    bad.append(os.path.join(dirpath, f))
    assert not bad, bad


def test_no_cpu_fallback():
    from hitgeom import dist_utils, model_seams, set_distance
    from hitgeom.pointnet2_ops import _ext

    x = torch.zeros(2, 16, 3)
    with pytest.raises(RuntimeError):
        set_distance.chamfer(x, x)
    with pytest.raises(RuntimeError):
        dist_utils.KNNDist()(x)
    with pytest.raises(RuntimeError):
        _ext.furthest_point_sampling(x, 4)
    with pytest.raises(RuntimeError):
        model_seams.square_distance(x, x)


def test_mirror_keeps_reference_signatures():
    from hitgeom import dist_utils as du
    from hitgeom import model_seams as ms
    from hitgeom import set_distance as sd
    from hitgeom.pointnet2_ops import _ext
    from hitgeom.pointnet2_ops import pointnet2_utils as pu

    def params(f):
        return list(inspect.signature(f).parameters)

    assert params(du.ChamferDist.__init__) == ["self", "method"]
    assert params(du.ChamferDist.forward) == ["self", "adv_pc", "ori_pc", "weights", "batch_avg"]
    assert params(du.HausdorffDist.forward) == ["self", "adv_pc", "ori_pc", "weights", "batch_avg"]
    assert params(du.KNNDist.__init__) == ["self", "k", "alpha"]
    assert params(du.KNNDist.forward) == ["self", "pc", "weights", "batch_avg"]
    assert params(du.ChamferkNNDist.__init__) == ["self", "chamfer_method", "knn_k", "knn_alpha", "chamfer_weight",
                                                  "knn_weight"]
    assert params(sd.ChamferDistance.forward) == ["self", "preds", "gts"]
    assert isinstance(sd.chamfer, sd.ChamferDistance) and isinstance(sd.hausdorff, sd.HausdorffDistance)
    assert params(ms.query_ball_point) == ["radius", "nsample", "xyz", "new_xyz"]
    assert params(ms.farthest_point_sample) == ["xyz", "npoint"]
    assert params(ms.knn) == ["x", "k"]
    for name in ("gather_points", "gather_points_grad", "furthest_point_sampling", "three_nn", "three_interpolate",
                 "three_interpolate_grad", "ball_query", "group_points", "group_points_grad"):
        assert callable(getattr(_ext, name)), name  # bindings.cpp:6-19
    assert params(_ext.ball_query) == ["new_xyz", "xyz", "radius", "nsample"]
    for name in ("furthest_point_sample", "gather_operation", "three_nn", "three_interpolate", "grouping_operation",
                 "ball_query", "QueryAndGroup", "GroupAll"):
        assert hasattr(pu, name), name


def test_install_registers_reference_import_names():
    import sys

    import hitgeom

    saved = {k: sys.modules.get(k) for k in ("pointnet2_ops", "pointnet2_ops._ext", "pytorch3d", "pytorch3d.ops")}
    try:
        for k in saved:
            sys.modules.pop(k, None)
        hitgeom.install()
        import pointnet2_ops._ext as e  # the reference's own import line (pointnet2_utils.py:8)
        from pytorch3d.ops import knn_gather, knn_points  # util/dist_utils.py:12

        assert callable(e.ball_query) and callable(knn_points) and callable(knn_gather)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
