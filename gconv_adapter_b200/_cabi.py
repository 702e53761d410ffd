"""ctypes binding of libgca.so (the C ABI declared in include/gca.h).

There is no CPU or PyTorch fallback: if the library has not been built
(``python -m gconv_adapter_b200.build``) every entry point raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import logging
import os
import threading

log = logging.getLogger("gconv_adapter_b200")

from . import build as _build

# The library file name carries the hash of the sources it was built from (gconv_adapter_b200/build.py), so a binary
# of older sources is never loaded.  GCA_LIB_PATH selects an alternative build (profiling experiments only).
LIB_PATH = os.environ.get("GCA_LIB_PATH") or _build.lib_path()
ABI_VERSION = 2

GCA_OK = 0
GCA_ERR_INDEX_RANGE = -4
GCA_ERR_UNSUPPORTED = -5
ACT = {"none": 0, "relu": 1, "silu": 2}

_f = C.c_void_p       # device pointers travel as integers
_i32, _i64, _sz = C.c_int32, C.c_int64, C.c_size_t


MAX_PEERS = 8
IPC_HANDLE_BYTES = 64


class Push(C.Structure):
    """gca_push: peer-mapped destinations that receive the rows a producing phase writes (include/gca.h)."""
    _fields_ = [("count", _i32), ("reserved", _i32), ("dst", C.c_void_p * MAX_PEERS)]


class PeerSync(C.Structure):
    """gca_peer_sync: the flag arrays of all GPUs of the group + the local sequence counter."""
    _fields_ = [("world", _i32), ("rank", _i32), ("flags", C.c_void_p * MAX_PEERS), ("seq", C.c_void_p)]


class GraphView(C.Structure):
    _fields_ = [("N", _i32), ("row_begin", _i32), ("row_end", _i32), ("normalize", _i32),
                ("capacity", _i64), ("rowptr", _f), ("colidx", _f), ("rowptr_t", _f), ("colidx_t", _f), ("dis", _f)]


# name -> (restype, argtypes); must list every symbol include/gca.h declares.
SIGNATURES = {
    "gca_abi_version": (C.c_int, []),
    "gca_status_string": (C.c_char_p, [C.c_int]),
    "gca_last_cuda_error": (C.c_char_p, []),
    "gca_shape_is_fast": (C.c_int, [_i32, _i32]),
    "gca_graph_workspace_bytes": (_sz, [_i64, _i32, _i32, _i32]),
    "gca_graph_build": (C.c_int, [_f, _f, _i64, _i32, _i32, _i32, C.c_int, _f, _sz, _f, C.POINTER(C.c_void_p)]),
    "gca_graph_validate": (C.c_int, [_f, _f, C.POINTER(_i64), C.POINTER(_i64)]),
    "gca_graph_validate_async": (C.c_int, [_f, _f, _f]),
    "gca_graph_validate_finish": (C.c_int, [_f, _f, C.POINTER(_i64), C.POINTER(_i64)]),
    "gca_graph_destroy": (None, [_f]),
    "gca_graph_get_view": (C.c_int, [_f, C.POINTER(GraphView)]),
    "gca_graph_edge_coef": (C.c_int, [_f, _f, _f]),
    "gca_hub_scratch_bytes": (_sz, [_f]),
    "gca_hub_scratch_bytes_r": (_sz, [_f, _i32]),
    "gca_propagate": (C.c_int, [_f, C.c_int, _f, _i64, _f, _i64, _f, _f, _i32, _f]),
    "gca_fwd_project": (C.c_int, [_f, _f, _i64, _f, _f, C.POINTER(Push), _i32, _i32, _f]),
    "gca_fwd_hop1": (C.c_int, [_f, _f, _f, C.c_int, _f, _f, _f, C.POINTER(Push), _i32, _f]),
    "gca_fwd_hop2_up": (C.c_int, [_f, _f, _f, _i64, _f, _f, _f, C.c_int, _f, _f, _i64, _f, _i32, _i32, _f]),
    "gca_fwd_hop2_up_add": (C.c_int, [_f, _f, _f, _i64, _f, _f, _f, C.c_int, _f, _f, _i64, _f, _i64, _f, _i32, _i32, _f]),
    "gca_bwd_scratch_bytes": (_sz, [_i32, _i32]),
    "gca_bwd_up": (C.c_int, [_f, _f, _i64, _f, _f, _f, _f, _f, C.POINTER(Push), _i32, _i32, _f]),
    "gca_bwd_up_project": (C.c_int, [_f, _f, _i64, _f, _f, _f, _f, C.POINTER(Push), _i32, _i32, _f]),
    "gca_bwd_up_wgrad": (C.c_int, [_f, _f, _i64, _f, _f, _i32, _i32, _f]),
    "gca_bwd_hop2": (C.c_int, [_f, _f, _f, _f, C.c_int, _f, _f, _f, C.POINTER(Push), _i32, _f]),
    "gca_bwd_hop1_down": (C.c_int, [_f, _f, _f, _i64, _f, _i64, _f, _f, C.c_int, _f, _f, _i64, _f, _f, _i32, _i32, _f]),
    "gca_bwd_finalize": (C.c_int, [_f, _f, _f, _f, C.c_int, _f, _f, _f, _f, _f, _i32, _i32, _f]),
    "gca_forward_workspace_bytes": (_sz, [_f, _i32, _i32]),
    "gca_forward": (C.c_int, [_f, _f, _i64, _f, _f, _f, _f, _f, C.c_int, C.c_int, _f, _f, _f, _f, _f, _i64, _i32, _i32, _f]),
    "gca_forward_add": (C.c_int, [_f, _f, _i64, _f, _f, _f, _f, _f, C.c_int, C.c_int, _f, _f, _f, _f, _f, _i64, _f, _i64,
                                  _i32, _i32, _f]),
    "gca_backward_workspace_bytes": (_sz, [_f, _i32, _i32]),
    "gca_backward": (C.c_int, [_f, _f, _i64, _f, _i64, _f, _f, _f, _f, _f, _f, _f, C.c_int, C.c_int, _f,
                               _f, _i64, _f, _f, _f, _f, _f, _i32, _i32, _f]),
    "gca_peer_barrier": (C.c_int, [C.POINTER(PeerSync), _f]),
    "gca_peer_allreduce": (C.c_int, [C.POINTER(PeerSync), C.POINTER(Push), _f, _f, _i32, _f]),
    "gca_push_rows": (C.c_int, [_f, _i64, C.POINTER(Push), _f]),
    "gca_peer_alloc": (C.c_int, [_sz, C.POINTER(C.c_void_p)]),
    "gca_peer_free": (C.c_int, [_f]),
    "gca_peer_export": (C.c_int, [_f, C.c_char_p]),
    "gca_peer_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "gca_peer_close": (C.c_int, [_f]),
    "gca_layernorm_scratch_bytes": (_sz, [_i32]),
    "gca_layernorm_scale_fwd": (C.c_int, [_f, _i64, _f, _f, _f, C.c_float, _f, _i64, _f, _f, _i32, _i32, _f]),
    "gca_layernorm_scale_add_fwd": (C.c_int, [_f, _i64, _f, _f, _f, C.c_float, _f, _i64, _f, _i64, _f, _f, _i32, _i32, _f]),
    "gca_layernorm_scale_bwd": (C.c_int, [_f, _i64, _f, _i64, _f, _f, _f, _f, _f, _f, _i64, _f, _f, _f, _f, _i32, _i32, _f]),
    "gca_batchnorm_scratch_bytes": (_sz, [_i32]),
    "gca_batchnorm_scale_fwd": (C.c_int, [_f, _i64, _f, _f, _f, C.c_float, C.c_int, C.c_float, _f, _f, _f, _i64, _f, _f, _f,
                                          _i32, _i32, _f]),
    "gca_batchnorm_scale_bwd": (C.c_int, [_f, _i64, _f, _i64, _f, _f, _f, _f, _f, C.c_int, _f, _i64, _f, _f, _f, _f, _i32, _i32,
                                          _f]),
    "gca_nccl_available": (C.c_int, []),
    "gca_forward_nccl_workspace_bytes": (_sz, [_f, _i32, _i32, _i32]),
    "gca_forward_nccl": (C.c_int, [_f, _f, _i32, _i32, _f, _i64, _f, _f, _f, _f, _f, C.c_int, C.c_int, _f, _f, _f, _f, _f, _i64,
                                   _i32, _i32, _f]),
    "gca_backward_nccl_workspace_bytes": (_sz, [_f, _i32, _i32, _i32]),
    "gca_backward_nccl": (C.c_int, [_f, _f, _i32, _i32, _f, _i64, _f, _i64, _f, _f, _f, _f, _f, _f, _f, C.c_int, C.c_int, _f,
                                    _f, _i64, _f, _f, _f, _f, _f, _i32, _i32, _f]),
    "gca_launch_count": (_i64, []),
    "gca_profile_enable": (C.c_int, [C.c_int]),
    "gca_profile_report": (C.c_int, [C.c_char_p, _sz]),
}

_lib = None
_lock = threading.Lock()


def load():
    """Load libgca.so once; raise loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.isfile(LIB_PATH):
                raise RuntimeError(
                    f"gconv_adapter_b200: CUDA library not built for these sources ({LIB_PATH} missing). "
                    "Run `python -m gconv_adapter_b200.build` (needs nvcc); there is no CPU fallback.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            if lib.gca_abi_version() != ABI_VERSION:
                raise RuntimeError("gconv_adapter_b200: libgca.so ABI version mismatch; rebuild it")
            _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    """Turn a negative gca_status into RuntimeError (and log it: the reference's inductive
    training loop swallows RuntimeError and skips the batch,
    /root/reference/scripts/finetune_inductive_learning.py:51-53)."""
    if status == GCA_OK:
        return
    lib = load()
    msg = f"{what}: {lib.gca_status_string(status).decode()}"
    if status == -3:
        msg += f" ({lib.gca_last_cuda_error().decode()})"
    log.error("gconv_adapter_b200 %s", msg)
    raise RuntimeError("gconv_adapter_b200 " + msg)
