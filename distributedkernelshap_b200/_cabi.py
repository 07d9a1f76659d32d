"""ctypes binding of the C ABI in ``include/dks.h`` (``libdks.so``).

This is the reference-side stub a maintainer would add (INTEGRATION.md): plain pointers and sizes, torch
tensors appear only as ``data_ptr()`` integers.  Loading fails loudly when the library is absent; there is
no alternative implementation to fall back to.
"""
import ctypes as C
import os

from . import build as _build

_lib = None

c_double_p = C.POINTER(C.c_double)
c_u64_p = C.POINTER(C.c_uint64)
c_i32_p = C.POINTER(C.c_int32)

DKS_OK = 0
DKS_ERR_INVALID = 1
DKS_ERR_CUDA = 2
DKS_ERR_UNSUPPORTED = 3
DKS_ERR_PLAN_MISSING = 4
DKS_ERR_NUMERIC = 5

ACT_IDENTITY = 0
ACT_BINARY_LOGISTIC = 1
ACT_SOFTMAX = 2
LINK_IDENTITY = 0
LINK_LOGIT = 1
KERNEL_AUTO = 0
KERNEL_SIMT = 1
KERNEL_TCGEN05 = 2
KERNEL_SHARED = 3

# name -> (restype, argtypes); every symbol include/dks.h declares
SIGNATURES = {
    "dks_version": (C.c_int, []),
    "dks_last_error": (C.c_char_p, []),
    "dks_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "dks_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "dks_destroy": (C.c_int, [C.c_void_p]),
    "dks_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dks_synchronize": (C.c_int, [C.c_void_p]),
    "dks_set_background": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "dks_set_groups": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "dks_set_model": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_int]),
    "dks_set_mlp_model": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                    C.c_double, C.c_int]),
    "dks_set_link": (C.c_int, [C.c_void_p, C.c_int]),
    "dks_fit": (C.c_int, [C.c_void_p]),
    "dks_num_outputs": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dks_get_fnull": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dks_predict_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dks_set_nsamples": (C.c_int, [C.c_void_p, C.c_int]),
    "dks_effective_nsamples": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "dks_set_shared_plan": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "dks_set_plan_projection": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "dks_clear_plans": (C.c_int, [C.c_void_p]),
    "dks_has_shared_plan": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int)]),
    "dks_set_l1": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "dks_set_l1_tables": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 8 + [C.c_double, C.c_double, C.c_int]),
    "dks_set_plan_sampling": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double]),
    "dks_set_plan_mode": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64]),
    "dks_set_row_offset": (C.c_int, [C.c_void_p, C.c_int64]),
    "dks_get_instance_plans": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "dks_prepare_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dks_prepare_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dks_get_m_histogram": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dks_run_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "dks_set_peers": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64]),
    "dks_set_peer_flags": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dks_graph_launches": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dks_get_link_fx": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "dks_get_varying": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dks_explain_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "dks_explain_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "dks_summarise_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dks_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    "dks_host_free": (C.c_int, [C.c_void_p]),
    "dks_last_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "dks_set_kernel": (C.c_int, [C.c_void_p, C.c_int]),
    "dks_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "dks_kernel_launches": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dks_last_timings": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dks_debug_score_dump": (C.c_int, [C.c_void_p, C.c_int]),
    "dks_debug_get_timeline": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dks_debug_get_scores": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}


class DksError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libdks error {code}: {message}")
        self.code = code


def load(build_if_needed=True):
    """Load libdks.so (building it first when stale and nvcc is available).  Raises if it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("DKS_LIB", _build.LIB_PATH)     # DKS_LIB: tuning variants built by scripts/build_variants.sh
    if path == _build.LIB_PATH and build_if_needed and _build.is_stale() and _build.find_nvcc() is not None:
        _build.build_library()
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: run `python -m distributedkernelshap_b200.build` "
                          "(there is no CPU fallback for the KernelSHAP hot path)")
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib


def check(rc):
    if rc != DKS_OK:
        msg = load().dks_last_error()
        raise DksError(rc, msg.decode() if msg else "")
    return rc


def ptr(arr):
    """Host pointer of a C-contiguous numpy array (or None)."""
    if arr is None:
        return None
    return arr.ctypes.data_as(C.c_void_p)
