"""Stage the UNMODIFIED reference Python tree: copy every `*.py` under $HITADV_REFERENCE (a TRLou/HiT-ADV checkout) into
`oracle/_ref/pytree/`, byte for byte.

TEST INFRASTRUCTURE ONLY.  `oracle/_ref/` is git-ignored (no reference source enters the history); copy it along to a
GPU machine that has no reference checkout, like `oracle/_ref/_ext_ref.so`.  The staged
tree lets `tests/test_gpu_unmodified_callers.py` run the reference's own attack classes (CW/kNN.py, CW/UKNN.py,
ShapeAttack/HiT_ADV.py) and its evaluation block (util/other_utils.py eval_ASR) ON A B200 over hitgeom's seams
(`hitgeom.install()` + `patch_reference()`), files unchanged.  Nothing in the product imports it.
"""
import os
import shutil

REF = os.environ.get("HITADV_REFERENCE", "")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "pytree")


def stage():
    if not REF or not os.path.isdir(REF):
        return OUT if os.path.isdir(OUT) else None
    n = 0
    for root, dirs, files in os.walk(REF):
        dirs[:] = [d for d in dirs if d not in ("__pycache__", ".git", "_ext-src")]
        for f in files:
            if not f.endswith(".py"):
                continue
            src = os.path.join(root, f)
            dst = os.path.join(OUT, os.path.relpath(src, REF))
            os.makedirs(os.path.dirname(dst), exist_ok=True)
            if not os.path.exists(dst) or open(dst, "rb").read() != open(src, "rb").read():
                shutil.copyfile(src, dst)
            n += 1
    with open(os.path.join(OUT, "STAGED_FROM"), "w") as fh:
        fh.write(f"{REF}: {n} python files, unmodified (oracle/stage_ref.py)\n")
    return OUT


if __name__ == "__main__":
    print(stage())
