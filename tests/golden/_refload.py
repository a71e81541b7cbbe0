"""Load the UNMODIFIED reference from $HITADV_REFERENCE (a checkout of TRLou/HiT-ADV) for golden-vector generation.

Only the `make_golden*.py` scripts import this: the reference is not part of the repository, so nothing under `tests/test_*.py`, `bench.py` or `__graft_entry__.py` may import it.

What is patched (harness-side only, the reference files are read-only and untouched):
  * stub modules for the reference's absent third-party imports (`pytorch3d`, `mayavi`, `open3d`,
    `matplotlib`, `seaborn`) -- SURVEY.md R6;
  * `Tensor.cuda` / `Module.cuda` become identity so that the loss classes, which hard-code
    `.cuda()` (`util/dist_utils.py:36,76,115,171`), run on this CPU-only box -- SURVEY.md R5.
"""
import importlib
import os
import importlib.util
import sys
import types

REF = os.environ.get("HITADV_REFERENCE", "")


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_stubs():
    import torch

    sys.dont_write_bytecode = True

    def _unavailable(*a, **k):
        raise RuntimeError("pytorch3d is not installed; golden vectors never touch it")

    p3d = _stub("pytorch3d")
    p3d.ops = _stub("pytorch3d.ops", knn_points=_unavailable, knn_gather=_unavailable)
    p3d.loss = _stub("pytorch3d.loss", chamfer_distance=_unavailable)
    mv = _stub("mayavi")
    mv.mlab = _stub("mayavi.mlab")
    _stub("open3d")
    mpl = _stub("matplotlib", use=lambda *a, **k: None)
    mpl.pyplot = _stub("matplotlib.pyplot")
    _stub("seaborn", set=lambda *a, **k: None)
    torch.Tensor.cuda = lambda self, *a, **k: self
    torch.nn.Module.cuda = lambda self, *a, **k: self
    if REF not in sys.path:
        sys.path.insert(0, REF)


def by_path(modname, relpath):
    """Import one reference file by path, bypassing its package `__init__` (SURVEY.md section 8c)."""
    spec = importlib.util.spec_from_file_location(modname, f"{REF}/{relpath}")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load():
    """Returns a namespace with the reference modules the hot path consists of."""
    install_stubs()
    ns = types.SimpleNamespace()
    ns.set_distance = by_path("ref_set_distance", "util/set_distance.py")
    ns.dist_utils = importlib.import_module("util.dist_utils")
    ns.pn2_utils = by_path("ref_model_pointnet2_utils", "model/pointnet2_utils.py")
    ns.dgcnn = by_path("ref_model_dgcnn", "model/dgcnn_cls.py")
    return ns
