"""Compile the UNMODIFIED reference `pointnet2_ops._ext` (the nine CUDA kernels of SURVEY.md section 2.2)
for sm_100 into `oracle/_ref/`, straight from the sources where they lie under $HITADV_REFERENCE.

TEST INFRASTRUCTURE ONLY.  The resulting `oracle/_ref/_ext_ref.so` is the GPU-side oracle for the
pointnet2_ops rows (a12-a17): `tests/test_gpu_pointnet2_ref.py` compares the hitgeom kernels against it
on the same inputs.  It is never imported by the product package, `oracle/_ref/` is git-ignored (no
reference code enters history) but it does travel to the GPU box with the gpurun snapshot.

The only thing changed w.r.t. the reference's own build (`pointnet2_ops_lib/setup.py:19`) is the arch
list, which upstream pins to sm_37..sm_75 (SURVEY.md R15).  No reference source is copied or edited.

Runs only where $HITADV_REFERENCE names a reference checkout; elsewhere a prebuilt .so is used if present.
"""
import glob
import os
import sys

REF_SRC = os.path.join(os.environ.get("HITADV_REFERENCE", "/nonexistent"), "pointnet2_ops_lib/pointnet2_ops/_ext-src")
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def build(verbose=False):
    if not os.path.isdir(REF_SRC):
        return None
    so = os.path.join(OUT, "_ext_ref.so")
    if os.path.exists(so):
        return so
    os.makedirs(OUT, exist_ok=True)
    os.environ["TORCH_CUDA_ARCH_LIST"] = "10.0"
    from torch.utils.cpp_extension import load

    srcs = sorted(glob.glob(f"{REF_SRC}/src/*.cpp") + glob.glob(f"{REF_SRC}/src/*.cu"))
    load(
        "_ext_ref",
        sources=srcs,
        extra_include_paths=[f"{REF_SRC}/include"],
        extra_cflags=["-O3"],
        extra_cuda_cflags=["-O3", "-lineinfo"],
        build_directory=OUT,
        with_cuda=True,
        is_python_module=True,
        verbose=verbose,
    )
    return so if os.path.exists(so) else None


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv))
