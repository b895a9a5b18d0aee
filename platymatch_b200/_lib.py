"""ctypes binding of libplatymatch_b200.so (C ABI declared in include/platymatch_b200.h).

There is no CPU fallback: if the shared library is missing, or a compute entry point is called
without a CUDA device, this module raises.  torch is used only for device memory and streams.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libplatymatch_b200.so")

NBINS = 360
LAP_STATS = 16
# PM_LAP_STAT_* slots of the assignment's statistics that Python code reads by name
LAP_STAT = {"DIJKSTRA_STEPS": 3, "BIDS": 5, "REFRESHES": 6, "REFRESH_CYCLES": 9, "AUCTION_CYCLES": 10,
            "SAP_DENSE_RELAX": 12, "PATH": 13, "SAP_CYCLES": 14}
# PM_LAP_PATH_* bits of the assignment's `path` statistic (PM_LAP_STAT_PATH): which kernels a solve ran
LAP_PATH = {"SQUARED": 1, "SPARSE_AUCTION": 2, "DENSE_AUCTION": 4, "SAP_SPARSE": 8, "SAP_DENSE8": 16,
            "SAP_DENSE16": 32, "SAP_DENSE24": 64, "RING_SMEM": 128}
CHI2_EPS = 2.0 ** -60
CHI2_TILE = 128
TRANSFORMS = {"Affine": 0, "Similar": 1}      # PM_TRANSFORM_* (the widget's strings, _dock_widget.py:627)
VOLUME_DTYPES = {"int32": 0, "uint16": 1, "float32": 2}    # PM_LABEL_I32, PM_LABEL_U16, PM_RESAMPLE_F32

_vp, _i, _d, _sz, _u64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_double, ctypes.c_size_t, ctypes.c_ulonglong

# name -> (restype, argtypes); must list every symbol the header declares (tests/test_abi.py checks)
SIGNATURES = {
    "pm_version": (_i, []),
    "pm_last_error_string": (ctypes.c_char_p, []),
    "pm_device_count": (_i, []),
    "pm_sm_count": (_i, [_i]),
    "pm_launch_count": (_u64, []),
    "pm_probe_fp32_fma": (_i, [_i, _i, _vp, _vp, _vp]),
    "pm_label_max_id": (_i, [_vp, _i, _sz, _vp, _vp]),
    "pm_label_workspace_bytes": (_sz, [ctypes.c_uint32]),
    "pm_label_centroids": (_i, [_vp, _i, _i, _i, _i, ctypes.c_uint32, _d, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pm_resample_affine": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _d, _vp, _i, _i, _i, _vp]),
    "pm_detect_pass": (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, ctypes.c_float, _vp, _vp]),
    "pm_detect_otsu_workspace_bytes": (_sz, []),
    "pm_detect_otsu": (_i, [_vp, _sz, _d, _vp, _vp, _sz, _vp]),
    "pm_detect_minima": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, ctypes.c_longlong, _vp, _vp, _vp, _vp]),
    "pm_detect_suppress_workspace_bytes": (_sz, [ctypes.c_longlong, _i, _i, _i, _d, _d]),
    "pm_detect_suppress": (_i, [_vp, _vp, ctypes.c_longlong, _i, _i, _i, _vp, _d, _d, _d, _vp, _vp, _sz, _vp]),
    "pm_cdist": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp]),
    "pm_cloud_stats": (_i, [_vp, _i, _vp, _vp]),
    "pm_mean_distance_workspace_bytes": (_sz, [_i]),
    "pm_mean_distance": (_i, [_vp, _i, _vp, _vp, _sz, _vp]),
    "pm_shape_context_hist_rows": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "pm_chi2_operand": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "pm_chi2_operand_f32": (_i, [_vp, _i, _vp, _i, _vp, _vp]),
    "pm_chi2_cost": (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _vp, _i, _vp]),
    "pm_lap_workspace_bytes": (_sz, [_i, _i, _i]),
    "pm_lap_solve": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pm_ransac_workspace_bytes": (_sz, [_i]),
    "pm_ransac": (_i, [_vp, _vp, _i, _vp, _i, _i, _d, _u64, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pm_icp_workspace_bytes2": (_sz, [_i, _i]),
    "pm_icp": (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pm_fit_affine": (_i, [_vp, _vp, _i, _vp, _vp]),
    "pm_fit_similar": (_i, [_vp, _vp, _i, _vp, _vp]),
    "pm_select_best": (_i, [_vp, _vp, _i, _vp, _vp, _vp]),
    "pm_apply_affine": (_i, [_vp, _i, _vp, _vp, _vp]),
    "pm_gather_points": (_i, [_vp, _vp, _i, _vp, _vp]),
    "pm_compose": (_i, [_vp, _vp, _vp, _vp]),
    "pm_peer_alloc": (_i, [_sz, _vp]),
    "pm_peer_free": (_i, [_vp]),
    "pm_peer_export": (_i, [_vp, _vp]),
    "pm_peer_open": (_i, [_vp, _vp]),
    "pm_peer_close": (_i, [_vp]),
    "pm_host_mean_distance": (_i, [_vp, _i, _i, _vp]),
    "pm_host_shape_context": (_i, [_vp, _i, _vp, _d, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
}

_LIB = None


class PlatyMatchError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises ImportError loudly when it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "platymatch_b200: %s is missing - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C platymatch_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _LIB = lib
    return _LIB


def check(rc, what=""):
    """Map a C status to a Python exception (ValueError for bad arguments, as numpy callers expect)."""
    if rc == 0:
        return
    msg = load().pm_last_error_string().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError("%s: %s" % (what, msg))
    raise PlatyMatchError("%s failed (%d): %s" % (what, rc, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available() or load().pm_device_count() < 1:
        raise PlatyMatchError("platymatch_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


def ptr(t):
    """Device pointer of a torch tensor (or None -> NULL)."""
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
