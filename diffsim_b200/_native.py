"""ctypes binding of libdiffsim_b200.so (the C ABI declared in include/diffsim_b200.h).

There is no fallback: if the shared library is missing, or a compute entry point
fails (no sm_100 GPU, bad arguments), an exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# DIFFSIM_B200_LIB selects another build of the same library (e.g. the -DDS_TRACE debug build)
LIB_PATH = os.environ.get("DIFFSIM_B200_LIB") or os.path.join(_HERE, "_lib", "libdiffsim_b200.so")

DS_OK = 0
DS_ERR_INVALID, DS_ERR_UNSUPPORTED, DS_ERR_CUDA, DS_ERR_WORKSPACE = -1, -2, -3, -4
DS_F16, DS_BF16, DS_F32 = 0, 1, 2
DS_SIM_COSINE, DS_SIM_MSE, DS_SIM_MINMAX_COSINE = 0, 1, 2
DS_OPT_ROUND_SCORES = 1

_ERR_NAMES = {
    DS_ERR_INVALID: "DS_ERR_INVALID",
    DS_ERR_UNSUPPORTED: "DS_ERR_UNSUPPORTED",
    DS_ERR_CUDA: "DS_ERR_CUDA",
    DS_ERR_WORKSPACE: "DS_ERR_WORKSPACE",
}


class DiffSimError(RuntimeError):
    """A ds_* entry point returned a negative status."""

    def __init__(self, code: int, message: str):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {message}")
        self.code = code


class Tensor4(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("size", C.c_int64 * 4), ("stride", C.c_int64 * 4), ("dtype", C.c_int32)]


class Tensor5(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("size", C.c_int64 * 5), ("stride", C.c_int64 * 5), ("dtype", C.c_int32)]


# name -> (restype, argtypes); every symbol include/diffsim_b200.h declares
_i64, _vp, _sz, _f, _i = C.c_int64, C.c_void_p, C.c_size_t, C.c_float, C.c_int
PROTOTYPES = {
    "ds_abi_version": (_i, []),
    "ds_last_error": (C.c_char_p, []),
    "ds_device_ok": (_i, []),
    "ds_profile_enable": (_i, [_i]),
    "ds_profile_collect": (_i, [C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "ds_debug_set_trace": (_i, [_vp, _i]),
    "ds_debug_set_gemm_variant": (_i, [_i]),
    "ds_debug_set_simmat_blocked": (_i, [_i]),
    "ds_debug_set_attn_mc": (_i, [_i]),
    "ds_attn_fwd": (_i, [Tensor4, Tensor4, Tensor4, _f, Tensor4, _vp, _sz, _vp]),
    "ds_attn_fwd_workspace_bytes": (_sz, [Tensor4, Tensor4]),
    "ds_attn_bwd": (_i, [Tensor4, Tensor4, Tensor4, Tensor4, Tensor4, _f, Tensor4, Tensor4, Tensor4, _vp, _sz, _vp]),
    "ds_attn_bwd_workspace_bytes": (_sz, [Tensor4, Tensor4]),
    "ds_aas_dir_bwd": (_i, [Tensor4, Tensor4, Tensor4, Tensor4, Tensor4, _f, _i, _vp, Tensor4, Tensor4, Tensor4, Tensor4,
                            Tensor4, _vp, _sz, _vp]),
    "ds_aas_dir_bwd_workspace_bytes": (_sz, [Tensor4, Tensor4]),
    "ds_aas_groups_bwd": (_i, [Tensor5, Tensor5, Tensor5, Tensor5, Tensor5, _vp, _vp, _i64, _vp, _i64, _f, _i, _vp, Tensor5,
                               Tensor5, Tensor5, Tensor5, Tensor5, _vp, _sz, _vp]),
    "ds_aas_groups_bwd_workspace_bytes": (_sz, [Tensor5, Tensor5, _i64, _i64]),
    "ds_aas_pairs_bwd": (_i, [Tensor5, Tensor5, Tensor5, _vp, _i64, _f, _i, _vp, Tensor5, Tensor5, Tensor5, _vp, _sz, _vp]),
    "ds_aas_pairs_bwd_workspace_bytes": (_sz, [Tensor5, _i64]),
    "ds_aas_triplets_bwd": (_i, [Tensor5, Tensor5, Tensor5, _vp, _i64, _f, _i, _vp, _vp, Tensor5, Tensor5, Tensor5, _vp, _sz,
                                 _vp]),
    "ds_aas_triplets_bwd_workspace_bytes": (_sz, [Tensor5, _i64]),
    "ds_aas_matrix_bwd": (_i, [Tensor5, Tensor5, Tensor5, Tensor5, Tensor5, _f, _i, _vp, _i64, Tensor5, Tensor5, Tensor5,
                               Tensor5, Tensor5, _vp, _sz, _vp]),
    "ds_aas_matrix_bwd_workspace_bytes": (_sz, [Tensor5, Tensor5]),
    "ds_aas_groups": (_i, [Tensor5, Tensor5, Tensor5, Tensor5, Tensor5, _vp, _vp, _i64, _vp, _i64, _f, _i, _vp, _vp, _sz, _vp]),
    "ds_aas_groups_workspace_bytes": (_sz, [Tensor5, _i64, _i64]),
    "ds_aas_pairs": (_i, [Tensor5, Tensor5, Tensor5, _vp, _i64, _f, _i, _vp, _vp, _sz, _vp]),
    "ds_aas_pairs_workspace_bytes": (_sz, [Tensor5, _i64]),
    "ds_aas_triplets": (_i, [Tensor5, Tensor5, Tensor5, _vp, _i64, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "ds_aas_triplets_workspace_bytes": (_sz, [Tensor5, _i64]),
    "ds_aas_matrix": (_i, [Tensor5, Tensor5, Tensor5, Tensor5, Tensor5, _f, _i, _vp, _i64, _vp, _sz, _vp]),
    "ds_aas_matrix_workspace_bytes": (_sz, [Tensor5, Tensor5]),
    "ds_pair_reduce": (_i, [_vp, _vp, _i64, _i64, _i64, _i64, _i, _i, _vp, _vp, _sz, _vp]),
    "ds_pair_reduce_workspace_bytes": (_sz, [_i64, _i64]),
    "ds_pair_reduce_bwd": (_i, [_vp, _vp, _i64, _i64, _i64, _i64, _i, _i, _vp, _vp, _i64, _vp, _i64, _vp, _sz, _vp]),
    "ds_pair_reduce_bwd_workspace_bytes": (_sz, [_i64, _i64]),
    "ds_simmat": (_i, [_vp, _i64, _i64, _vp, _i64, _i64, _i64, _i, _i, _vp, _i64, _vp, _sz, _vp]),
    "ds_simmat_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "ds_qkv_project": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _i64, _i64, C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _i, _vp]),
    "ds_qkv_project_bwd": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, C.POINTER(C.c_void_p), C.POINTER(C.c_int64),
                                _vp, _i64, _vp, _i64, _vp, _i, _vp, _sz, _vp]),
    "ds_qkv_project_bwd_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64]),
    "ds_twoafc": (_i, [_vp, _vp, _i64, _i, _vp, _vp, _vp]),
}

_lib = None
_lock = threading.Lock()


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. "
                "Run `python -c 'import __graft_entry__ as g; g.build()'` (or diffsim_b200/csrc/build.sh). "
                "diffsim_b200 has no CPU or PyTorch fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        if lib.ds_abi_version() != 1:
            raise RuntimeError(f"ABI mismatch: library reports version {lib.ds_abi_version()}, binding expects 1")
        _lib = lib
        return lib


def last_error() -> str:
    msg = load().ds_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int) -> None:
    if rc != DS_OK:
        raise DiffSimError(rc, last_error())
