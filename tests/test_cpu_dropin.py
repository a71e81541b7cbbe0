"""Drop-in check against the UNMODIFIED reference tree, a checkout of TRLou/HiT-ADV named by $HITADV_REFERENCE (not part
of this repository: without it the test skips): with `hitgeom.install()` the reference's own modules import -- including its
pointnet2_ops wrapper, which would otherwise JIT-compile for sm_37..sm_75 -- `patch_reference()` rebinds the seams, and
every mirrored class / function has the reference's signature.  Runs in a subprocess (it rewires sys.modules)."""
import os
import subprocess
import sys
import tempfile
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("HITADV_REFERENCE", "")

SCRIPT = textwrap.dedent('''
    import inspect, sys, types
    sys.dont_write_bytecode = True
    sys.path.insert(0, "%(root)s/hit-adv_b200")
    sys.path.insert(0, "%(ref)s")
    sys.path.insert(0, "%(ref)s/pointnet2_ops_lib")
    # packages the reference imports for plotting / IO that are not installed here (not part of the hot path)
    for name in ("mayavi", "mayavi.mlab", "open3d", "matplotlib", "matplotlib.pyplot", "seaborn", "h5py"):
        m = types.ModuleType(name); sys.modules[name] = m
    sys.modules["matplotlib"].use = lambda *a, **k: None
    sys.modules["seaborn"].set = lambda *a, **k: None
    import hitgeom
    hitgeom.install()
    import pointnet2_ops.pointnet2_utils as ref_pu          # the reference file, importing hitgeom's _ext
    assert ref_pu.__file__.startswith("%(ref)s"), ref_pu.__file__
    assert ref_pu._ext is sys.modules["pointnet2_ops._ext"]
    from util import dist_utils as ref_du, set_distance as ref_sd
    from model import pointnet2_utils as ref_mpu, dgcnn_cls as ref_dg
    patched = hitgeom.patch_reference()
    assert {"util.set_distance", "util.dist_utils", "model.pointnet2_utils", "model.dgcnn_cls"} <= set(patched), patched
    from hitgeom import dist_utils as du, model_seams as ms, set_distance as sd
    assert ref_du.ChamferDist.forward is du.ChamferDist.forward and ref_du.KNNDist.forward is du.KNNDist.forward
    assert ref_du.ChamferkNNDist.forward is du.ChamferkNNDist.forward and ref_sd.chamfer is sd.chamfer
    assert ref_mpu.farthest_point_sample is ms.farthest_point_sample and ref_mpu.query_ball_point is ms.query_ball_point
    assert ref_dg.knn is ms.knn and ref_dg.get_graph_feature is ms.get_graph_feature

    def same_signature(a, b):
        pa, pb = inspect.signature(a).parameters, inspect.signature(b).parameters
        assert list(pa) == list(pb), (a, list(pa), list(pb))
        for k in pa:
            assert pa[k].default == pb[k].default or (pa[k].default is pb[k].default), (a, k)

    import importlib
    orig_du = importlib.reload(importlib.import_module("util.dist_utils"))   # the reference's own definitions again
    for cls in ("ChamferDist", "HausdorffDist", "KNNDist", "ChamferkNNDist", "L2Dist"):
        same_signature(getattr(orig_du, cls).__init__, getattr(du, cls).__init__)
        same_signature(getattr(orig_du, cls).forward, getattr(du, cls).forward)
    from hitgeom import eval_metrics as em, clip_utils as cu, adv_utils as au, cw_knn
    same_signature(orig_du.CurvStdDist.forward, em.CurvStdDist.forward)
    import util.clip_utils as ref_cu, util.adv_utils as ref_au
    for cls in ("ClipPointsL2", "ClipPointsLinf", "ProjectInnerPoints", "ProjectInnerClipLinf"):
        same_signature(getattr(ref_cu, cls).forward, getattr(cu, cls).forward)
    for cls in ("LogitsAdvLoss", "UntargetedLogitsAdvLoss", "CrossEntropyAdvLoss"):
        same_signature(getattr(ref_au, cls).forward, getattr(au, cls).forward)
    orig_mpu = importlib.reload(importlib.import_module("model.pointnet2_utils"))
    for fn in ("square_distance", "index_points", "farthest_point_sample", "query_ball_point"):
        same_signature(getattr(orig_mpu, fn), getattr(ms, fn))
    orig_dg = importlib.reload(importlib.import_module("model.dgcnn_cls"))
    same_signature(orig_dg.knn, ms.knn)
    same_signature(orig_dg.get_graph_feature, ms.get_graph_feature)
    from CW.kNN import CWKNN as RefCWKNN
    from CW.UKNN import CWUKNN as RefCWUKNN
    ref_args = list(inspect.signature(RefCWKNN.__init__).parameters)
    assert list(inspect.signature(cw_knn.CWKNN.__init__).parameters)[:len(ref_args)] == ref_args
    ref_args = list(inspect.signature(RefCWUKNN.__init__).parameters)
    mine = list(inspect.signature(cw_knn.CWUKNN.__init__).parameters)
    assert mine[:len(ref_args)] == ref_args, (mine, ref_args)
    import pointnet2_ops.pointnet2_modules as ref_pm                        # reference modules over hitgeom's operators
    from hitgeom.pointnet2_ops import pointnet2_modules as pm
    for cls in ("PointnetSAModuleMSG", "PointnetSAModule", "PointnetFPModule"):
        same_signature(getattr(ref_pm, cls).__init__, getattr(pm, cls).__init__)
        same_signature(getattr(ref_pm, cls).forward, getattr(pm, cls).forward)
    # the callers: they import, find pytorch3d.ops / pointnet2_ops through hitgeom, and hitgeom's rebuilt versions keep
    # their constructor / call contracts
    sys.modules["matplotlib.pyplot"].figure = lambda *a, **k: None
    from ShapeAttack.HiT_ADV import HiT_ADV as RefHiT
    from hitgeom.hit_adv import HiT_ADV
    # the reference's parameters, in order, with its defaults; `graph=False` (CUDA-graph replay) is an optional extra
    pr, pm_ = inspect.signature(RefHiT.__init__).parameters, inspect.signature(HiT_ADV.__init__).parameters
    assert list(pm_)[:len(pr)] == list(pr) and list(pm_)[len(pr):] == ["graph"], (list(pr), list(pm_))
    assert all(pr[k].default == pm_[k].default for k in pr) and pm_["graph"].default is False
    same_signature(RefHiT.attack, HiT_ADV.attack)
    import FGM.GeoA3_args as ref_geo                                        # -> pointnet2_ops_lib.pointnet2_ops.pointnet2_utils
    assert ref_geo.pointnet2_utils._ext is sys.modules["pointnet2_ops._ext"]
    assert ref_geo.knn_points is sys.modules["pytorch3d.ops"].knn_points
    pa = list(inspect.signature(ref_geo.uniform_loss).parameters)
    assert list(inspect.signature(em.uniform_loss).parameters) == pa, pa
    same_signature(ref_geo.kNN_smoothing_loss, em.kNN_smoothing_loss)
    print("DROPIN_OK")
''')


@pytest.mark.skipif(not REF or not os.path.isdir(REF),
                    reason="needs the unmodified TRLou/HiT-ADV tree: set HITADV_REFERENCE to a checkout of it")
def test_unmodified_reference_imports_and_binds_to_hitgeom():
    out = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "ref": REF}], capture_output=True, text=True,
                         timeout=600, cwd=tempfile.gettempdir())
    assert out.returncode == 0 and "DROPIN_OK" in out.stdout, (out.stdout[-1500:], out.stderr[-3000:])
