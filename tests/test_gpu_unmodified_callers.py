"""The reference's OWN callers, files unchanged, executed on the B200 over hitgeom's seams.

`oracle/stage_ref.py` copies the reference's Python tree ($HITADV_REFERENCE, a checkout of TRLou/HiT-ADV; not part of
this repository) byte for byte into the git-ignored `oracle/_ref/pytree/`; without it the test skips.  A subprocess then puts that tree on sys.path, calls
`hitgeom.install()` (pointnet2_ops._ext and pytorch3d.ops resolve to hitgeom), imports the reference modules, calls
`hitgeom.patch_reference()` and runs, on CUDA:

  (a) `CW.kNN.CWKNN.attack` and `CW.UKNN.CWUKNN.attack` (CW/kNN.py:40-151, CW/UKNN.py) with the reference's own
      `ChamferkNNDist`, adversarial-loss and clip objects            -> tests/golden/cwknn_ref.npz
  (b) `ShapeAttack.HiT_ADV.HiT_ADV.attack` (HiT_ADV.py:44-287), 2 x 6 iterations   -> tests/golden/hitadv_ref.npz
  (c) `util.other_utils.eval_ASR` (other_utils.py:15-101): KNNDist(k=4), uniform_loss, CurvStdDist(k=4) and the ASR
      counters over two batches, with an attack object returning fixed clouds   -> tests/golden/evalasr_ref.npz

The golden files are outputs of the same unmodified classes on the build container's CPU.  Gates: (a) and (b) as for
hitgeom's native loops (statistical for CW-kNN, see tests/test_gpu_cwknn.py; 2e-3 + identical success count for
HiT-ADV); (c) ASR exact, metrics 1e-4 relative.  The subprocess also asserts that the reference classes really are
the staged files' and that the seams really are hitgeom's (no silent fall-through to the reference's torch path)."""
import os
import subprocess
import sys
import tempfile
import textwrap

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREE = os.path.join(ROOT, "oracle", "_ref", "pytree")

SCRIPT = textwrap.dedent('''
    import contextlib, io, logging, os, sys, tempfile, types
    sys.dont_write_bytecode = True
    ROOT, TREE = %(root)r, %(tree)r
    sys.path[:0] = [TREE, os.path.join(TREE, "pointnet2_ops_lib"), os.path.join(ROOT, "hit-adv_b200"), os.path.join(ROOT, "tests")]
    import numpy as np, torch
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    # packages the reference imports for plotting / IO that are not installed (not part of the hot path)
    for name in ("mayavi", "mayavi.mlab", "open3d", "matplotlib", "matplotlib.pyplot", "seaborn", "h5py", "pytorch3d.loss"):
        sys.modules[name] = types.ModuleType(name)
    sys.modules["matplotlib"].use = lambda *a, **k: None
    sys.modules["seaborn"].set = lambda *a, **k: None
    sys.modules["pytorch3d.loss"].chamfer_distance = None
    import hitgeom
    from hitgeom import _lib
    hitgeom.install()
    sys.modules["pytorch3d"].loss = sys.modules["pytorch3d.loss"]
    from util import dist_utils as ref_du, adv_utils as ref_au, clip_utils as ref_cu, other_utils as ref_ou
    from CW.kNN import CWKNN
    from CW.UKNN import CWUKNN
    from ShapeAttack.HiT_ADV import HiT_ADV
    for m in (ref_du, ref_ou, sys.modules["CW.kNN"], sys.modules["ShapeAttack.HiT_ADV"], sys.modules["FGM.GeoA3_args"]):
        assert m.__file__.startswith(TREE), m.__file__
    patched = hitgeom.patch_reference()
    assert {"util.set_distance", "util.dist_utils"} <= set(patched), patched
    from hitgeom import dist_utils as du
    assert ref_du.ChamferkNNDist.forward is du.ChamferkNNDist.forward and ref_du.KNNDist.forward is du.KNNDist.forward
    from util_models import TinyPointNet
    G = os.path.join(ROOT, "tests", "golden")
    hp_of = lambda g: {k[3:]: g[k].item() for k in g.files if k.startswith("hp_")}
    launches0 = _lib.launch_count()

    # ---- (a) CW-kNN attackers ----------------------------------------------------------------------------------
    g = np.load(os.path.join(G, "cwknn_ref.npz"))
    hp = hp_of(g)

    def check(adv, ref, pts, budget):
        assert adv.dtype == np.float32 and adv.shape == ref.shape
        assert np.abs(adv - pts).max() <= budget * (1 + 1e-6)
        err = np.abs(adv - ref)
        assert np.median(err) < 1e-5, np.median(err)
        assert (err > 1e-3).mean() < 0.10, (err > 1e-3).mean()

    model = TinyPointNet(40, seed=int(hp["model_seed"]))
    atk = CWKNN(model, ref_au.LogitsAdvLoss(kappa=hp["kappa"]), ref_du.ChamferkNNDist(),
                ref_cu.ClipPointsLinf(budget=hp["budget"]), attack_lr=hp["attack_lr"], num_iter=int(hp["num_iter"]))
    torch.manual_seed(int(hp["seed"]))
    with contextlib.redirect_stdout(io.StringIO()):
        adv, succ = atk.attack(torch.from_numpy(g["pts"]), torch.from_numpy(g["knn_target"]))
    check(adv, g["knn_adv"], g["pts"], hp["budget"])
    assert int(succ) == int(g["knn_success"]), (succ, g["knn_success"])
    atk = CWUKNN(model, ref_au.UntargetedLogitsAdvLoss(kappa=hp["kappa"]), ref_du.ChamferkNNDist(),
                 ref_cu.ProjectInnerClipLinf(budget=hp["budget"]), attack_lr=hp["attack_lr"], num_iter=int(hp["num_iter"]))
    torch.manual_seed(int(hp["seed"]))
    with contextlib.redirect_stdout(io.StringIO()):
        adv, succ = atk.attack(torch.from_numpy(np.concatenate([g["pts"], g["nrm"]], -1)), torch.from_numpy(g["label"]))
    check(adv, g["uknn_adv"], g["pts"], hp["budget"])
    assert int(succ) == int(g["uknn_success"])
    n_a = _lib.launch_count() - launches0
    assert n_a > 0, "the reference CW-kNN loop did not launch a single hitgeom kernel"
    print("CWKNN_OK", n_a)

    # ---- (b) HiT-ADV ---------------------------------------------------------------------------------------------
    g = np.load(os.path.join(G, "hitadv_ref.npz"))
    HP = hp_of(g)
    kappa = HP.pop("kappa")
    for k in ("binary_step", "num_iter", "curv_loss_knn", "central_num", "total_central_num"):
        HP[k] = int(HP[k])
    att = HiT_ADV(TinyPointNet(40, seed=int(g["model_seed"])), ref_au.UntargetedLogitsAdvLoss(kappa=kappa), clip_func=None, **HP)
    torch.manual_seed(int(g["seed"]))
    with contextlib.redirect_stdout(io.StringIO()):
        best, succ = att.attack(torch.from_numpy(g["data"]), torch.from_numpy(g["target"]))
    assert best.shape == g["best"].shape and int(succ) == int(g["success"]), (succ, g["success"])
    err = np.abs(best - g["best"]).max()
    assert err < 2e-3, err
    n_b = _lib.launch_count() - launches0 - n_a
    assert n_b > 0
    print("HITADV_OK", n_b, float(err))

    # ---- (c) eval_ASR's metric block ---------------------------------------------------------------------------
    g = np.load(os.path.join(G, "evalasr_ref.npz"))

    class FixedAttack:
        def __init__(self, advs):
            self.advs, self.i = advs, 0
        def attack(self, data, label):
            out = self.advs[self.i]; self.i += 1
            return out, None

    batches = [(torch.from_numpy(g[f"data{i}"]), torch.from_numpy(g[f"label{i}"])) for i in range(2)]
    args = types.SimpleNamespace(ker_weight=1.0, hide_weight=1.0, budget=0.55, max_sigm=1.2, min_sigm=0.1, central_num=192,
                                 attack_type="HiT_ADV", k=int(g["k"]), model="tiny")
    records = []
    class Grab(logging.Handler):
        def emit(self, record): records.append(record.getMessage())
    logging.getLogger().addHandler(Grab())
    tmp = tempfile.mkdtemp()
    os.makedirs(os.path.join(tmp, "log"))
    os.chdir(tmp)
    with contextlib.redirect_stdout(io.StringIO()):
        asr = ref_ou.eval_ASR(TinyPointNet(40, seed=int(g["model_seed"])).cuda(), batches, args, FixedAttack([g["adv0"], g["adv1"]]))
    vals = {}
    for m in records:
        for key, tag in (("knn", "Overall KNN dist: "), ("uniform", "Overall Uniform dist: "), ("curvstd", "Overall CurvStd dist: ")):
            if m.startswith(tag):
                vals[key] = float(m[len(tag):].replace("tensor(", "").replace(")", "").split(",")[0])
    assert abs(float(asr) - float(g["asr"])) < 1e-9, (asr, g["asr"])
    for key in ("knn", "uniform", "curvstd"):
        assert abs(vals[key] / float(g[key]) - 1) < 1e-4, (key, vals[key], float(g[key]))
    n_c = _lib.launch_count() - launches0 - n_a - n_b
    assert n_c > 0
    print("EVALASR_OK", n_c, vals)
    print("CALLERS_OK")
''')


@pytest.mark.skipif(not os.path.isdir(TREE), reason="needs the unmodified TRLou/HiT-ADV Python tree in oracle/_ref/pytree: "
                                                    "HITADV_REFERENCE=<checkout> python oracle/stage_ref.py")
def test_unmodified_reference_callers_run_on_cuda_over_hitgeom():
    out = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT, "tree": TREE}], capture_output=True, text=True,
                         timeout=900, cwd=tempfile.gettempdir())
    assert out.returncode == 0 and "CALLERS_OK" in out.stdout, (out.stdout[-2000:], out.stderr[-4000:])
    print(out.stdout[-600:])
