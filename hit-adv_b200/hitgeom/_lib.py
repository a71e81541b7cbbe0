"""ctypes binding of libhitgeom.so -- the C-ABI library declared in include/hitgeom.h.

There is NO CPU path and NO fallback: if the shared library is missing, or a tensor is not a contiguous
CUDA tensor of the expected dtype, the call raises.  PyTorch is used for device memory and streams only.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhitgeom.so")
CSRC = os.path.join(os.path.dirname(_HERE), "csrc")

_c_int, _c_float, _c_void_p, _c_size_t = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t

# name -> (restype, [argtypes]).  P = device pointer (void*), I = int, F = float, Z = size_t.
P, I, F, Z = _c_void_p, _c_int, _c_float, _c_size_t
_SIGNATURES = {
    "hg_version": (I, []),
    "hg_last_error": (ctypes.c_char_p, []),
    "hg_probe_fp32_peak": (I, [ctypes.POINTER(ctypes.c_float), P, P]),
    "hg_device_info": (I, [ctypes.POINTER(I), ctypes.POINTER(I), ctypes.POINTER(ctypes.c_longlong),
                           ctypes.POINTER(ctypes.c_longlong)]),
    "hg_nn_bidir_workspace_bytes": (Z, [I, I, I, I]),
    "hg_nn_bidir_f32": (I, [P, P, I, I, I, I, P, P, P, P, P, Z, P]),
    "hg_order_state_bytes": (Z, [I, I]),
    "hg_nn_bidir_temporal_f32": (I, [P, P, I, I, I, I, P, P, P, P, P, P, P, Z, P]),
    "hg_nn_bidir_tune": (None, [I, I]),
    "hg_knn_tune": (None, [I, I]),
    "hg_knn_force_shape": (None, [I, I]),
    "hg_knn_tune_small": (None, [I]),
    "hg_tune": (I, [ctypes.c_char_p, I]),
    "hg_prune_counters": (I, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "hg_prune_drain_counters": (I, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "hg_prune_order_counters": (I, [ctypes.POINTER(ctypes.c_ulonglong)]),
    "hg_launch_count": (ctypes.c_ulonglong, []),
    "hg_prof_enable": (None, [I]),
    "hg_prof_read": (I, [I, ctypes.POINTER(F), ctypes.POINTER(I)]),
    "hg_pairwise_dist_f32": (I, [P, P, I, I, I, I, P, P]),
    "hg_set_loss_f32": (I, [P, P, I, I, I, I, P, P, P, P, P]),
    "hg_set_loss_bwd_workspace_bytes": (Z, [I, I, I]),
    "hg_set_loss_bwd_f32": (I, [P, P, P, P, P, P, P, P, I, I, I, I, I, P, P, P, Z, P]),
    "hg_knn_self_workspace_bytes": (Z, [I, I, I, I]),
    "hg_knn_self_f32": (I, [P, I, I, I, I, P, P, P, Z, P]),
    "hg_knn_self_temporal_f32": (I, [P, I, I, I, I, P, P, P, I, P, Z, P]),
    "hg_knn_self_temporal_order_f32": (I, [P, I, I, I, I, P, P, P, I, P, P, Z, P]),
    "hg_knn_outlier_fwd_f32": (I, [P, I, I, I, F, P, P, P, P, P]),
    "hg_knn_outlier_bwd_workspace_bytes": (Z, [I, I, I]),
    "hg_knn_outlier_bwd_f32": (I, [P, P, P, P, I, I, I, I, P, P, Z, P]),
    "hg_knn_points_f32": (I, [P, P, I, I, I, I, P, P, P]),
    "hg_square_distance_f32": (I, [P, P, I, I, I, I, P, P]),
    "hg_fps_torch_f32": (I, [P, I, I, I, P, P, P]),
    "hg_query_ball_torch_f32": (I, [F, I, P, P, I, I, I, P, P]),
    "hg_index_points_f32": (I, [P, P, I, I, I, I, P, P]),
    "hg_index_points_grad_workspace_bytes": (Z, [I, I, I]),
    "hg_index_points_grad_f32": (I, [P, P, I, I, I, I, P, P, Z, P]),
    "hg_hitadv_deform_fwd_f32": (I, [P, P, P, P, I, I, I, P, P, P]),
    "hg_hitadv_deform_bwd_f32": (I, [P, P, P, P, P, P, P, I, I, I, P, P, P]),
    "hg_host_step_create": (P, [I, I, I]),
    "hg_host_step_destroy": (None, [P]),
    "hg_chamfer_knn_step_host_f32": (I, [P, P, P, I, I, I, F, F, F, P, P, P, P]),
    "hg_edge_feature_f32": (I, [P, P, I, I, I, I, P, P]),
    "hg_edge_feature_grad_workspace_bytes": (Z, [I, I, I]),
    "hg_edge_feature_grad_f32": (I, [P, P, I, I, I, I, P, P, Z, P]),
    "hg_p2_gather_points": (I, [I, I, I, I, P, P, P, P]),
    "hg_p2_scatter_workspace_bytes": (Z, [I, I, I]),
    "hg_p2_gather_points_grad": (I, [I, I, I, I, P, P, P, P, Z, P]),
    "hg_p2_furthest_point_sampling": (I, [I, I, I, P, P, P, P]),
    "hg_p2_ball_query": (I, [I, I, I, F, I, P, P, P, P]),
    "hg_p2_group_points": (I, [I, I, I, I, I, P, P, P, P]),
    "hg_p2_group_points_grad": (I, [I, I, I, I, I, P, P, P, P, Z, P]),
    "hg_p2_group_concat": (I, [I, I, I, I, I, P, P, P, P, P, P]),
    "hg_p2_group_concat_grad": (I, [I, I, I, I, I, P, P, P, P, P, Z, P]),
    "hg_p2_three_nn": (I, [I, I, I, P, P, P, P, P]),
    "hg_p2_three_interpolate": (I, [I, I, I, I, P, P, P, P, P]),
    "hg_p2_three_interpolate_grad": (I, [I, I, I, I, P, P, P, P, P, Z, P]),
}

_lib = None


class HitgeomError(RuntimeError):
    """Raised for every non-zero return code of the C ABI (bad arguments or a CUDA launch failure)."""


def build(verbose=False):
    """Compile libhitgeom.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
    import subprocess

    cmd = ["make", "-C", CSRC, "-j8"] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)
    return LIB_PATH


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: hitgeom has no CPU or PyTorch fallback. Build it with "
                f"`python -c 'import __graft_entry__ as g; g.build()'` or `make -C {CSRC}`.")
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here = header/library mismatch: fail loudly
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc, what):
    if rc != 0:
        msg = lib().hg_last_error().decode("utf-8", "replace")
        raise HitgeomError(f"{what} failed (code {rc}): {msg}")


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


def ptr(t):
    return t.data_ptr() if t is not None else None


def require(t, name, dtype=torch.float32, ndim=None):
    """The reference's CHECK_CUDA / CHECK_CONTIGUOUS / CHECK_IS_FLOAT|INT (_ext-src/include/utils.h:5-25)."""
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor")
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor (hitgeom has no CPU path)")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be a contiguous tensor")
    if t.dtype != dtype:
        raise RuntimeError(f"{name} must be a {dtype} tensor, got {t.dtype}")
    if ndim is not None and t.dim() != ndim:
        raise RuntimeError(f"{name} must have {ndim} dimensions, got shape {tuple(t.shape)}")
    return t


def workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


PROF_TAGS = {"nn_bidir": 0, "knn": 1, "fps": 2, "group": 3}


def prof_enable(on=True):
    lib().hg_prof_enable(1 if on else 0)


def prof_read(tag):
    """-> (summed device ms, launches) of the tagged hot kernel since prof_enable(True)."""
    ms, n = _c_float(), _c_int()
    check(lib().hg_prof_read(PROF_TAGS[tag], ctypes.byref(ms), ctypes.byref(n)), "hg_prof_read")
    return ms.value, n.value


def launch_count():
    return int(lib().hg_launch_count())


def probe_fp32_peak():
    """Measured FP32 FFMA throughput of the current device [TFLOP/s] (hg_probe_fp32_peak)."""
    out = _c_float()
    scratch = torch.zeros(4, dtype=torch.float32, device="cuda")
    check(lib().hg_probe_fp32_peak(ctypes.byref(out), scratch.data_ptr(), torch.cuda.current_stream().cuda_stream),
          "hg_probe_fp32_peak")
    return float(out.value)


def device_info():
    sm, clk = _c_int(), _c_int()
    l2, mem = ctypes.c_longlong(), ctypes.c_longlong()
    check(lib().hg_device_info(ctypes.byref(sm), ctypes.byref(clk), ctypes.byref(l2), ctypes.byref(mem)), "hg_device_info")
    return {"sm_count": sm.value, "clock_khz": clk.value, "l2_bytes": l2.value, "mem_bytes": mem.value}
