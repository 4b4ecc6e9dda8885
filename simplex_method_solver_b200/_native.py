"""ctypes binding of libspx_b200.so (C ABI declared in include/spx_b200.h).

There is no CPU fallback: if the library is missing or no CUDA device is
usable, every product entry point raises ``NativeUnavailable`` loudly.
PyTorch is used by the callers only to allocate device memory and to obtain
stream handles; nothing here takes or returns a torch type.
"""
from __future__ import annotations

import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libspx_b200.so")

ABI_VERSION = 8
LOOP_AUTO, LOOP_CLASSIC, LOOP_LOOKAHEAD, LOOP_RESIDENT, LOOP_FUSED = 0, 1, 2, 3, 4
LOOP_MODES = {None: LOOP_AUTO, "auto": LOOP_AUTO, False: LOOP_CLASSIC, "classic": LOOP_CLASSIC,
              True: LOOP_LOOKAHEAD, "lookahead": LOOP_LOOKAHEAD, "resident": LOOP_RESIDENT,
              "fused": LOOP_FUSED}
PIVOT, OPTIMAL, INCORRECT, NOCONV, CAP, PEER_TIMEOUT = 1, 0, -1, -2, -3, -4
RULE_REFERENCE, RULE_DANTZIG = 0, 1
# keys 1, 3, 4, 10 and 15 are retired (include/spx_b200.h)
OPT_TILED_MIN_BLOCKS, OPT_TILED_ROWS, OPT_FUSE_DEPTH = 2, 5, 6
OPT_FUSE_MIN_BLOCKS, OPT_FUSE_PRICING, OPT_FUSE_LOOKAHEAD, OPT_FUSE_TILE_ROWS, OPT_FUSE_PAIRS = 7, 8, 9, 11, 12
OPT_SHARD_THREADS, OPT_SHARD_CTAS, OPT_CLUSTER_SIZE = 13, 14, 16
RULES = {"reference": RULE_REFERENCE, "bland": RULE_REFERENCE, "dantzig": RULE_DANTZIG}
ENGINE_AUTO, ENGINE_SMEM, ENGINE_CLUSTER, ENGINE_GLOBAL, ENGINE_AUTO_GLOBAL = 0, 1, 2, 4, 5

# the two ValueError texts of pick_element(), /root/reference/src/simplex.py:89,139
ERROR_TEXT = {INCORRECT: "incorrect system", NOCONV: "simplex method does not converge"}


class NativeUnavailable(RuntimeError):
    pass


class SpxError(RuntimeError):
    pass


class SpxState(ctypes.Structure):
    """Mirror of ``spx_state`` (include/spx_b200.h), 128 bytes."""
    _fields_ = [
        ("status", ctypes.c_int32), ("r", ctypes.c_int32),
        ("c", ctypes.c_int64), ("p", ctypes.c_double),
        ("npiv", ctypes.c_int64), ("max_pivots", ctypes.c_int64),
        ("phase1", ctypes.c_int32), ("slot", ctypes.c_int32),
        ("hint_tag", ctypes.c_int64 * 2),
        ("hint_bneg", ctypes.c_int32 * 2), ("hint_fneg", ctypes.c_int32 * 2),
        ("reserved", ctypes.c_int64 * 6),
    ]


# name -> (restype, argtypes); every symbol include/spx_b200.h declares
_vp, _i32, _i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
_pi32, _pi64 = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
SIGNATURES = {
    "spx_version": (ctypes.c_int, []),
    "spx_last_error": (ctypes.c_char_p, []),
    "spx_ld": (_i64, [_i64]),
    "spx_cells": (_i64, [_i32, _i32]),
    "spx_colbuf_doubles": (_i64, [_i32]),
    "spx_state_bytes": (ctypes.c_int, []),
    "spx_device_info": (ctypes.c_int, [_pi32, _pi32, _pi32]),
    "spx_launch_count": (_i64, [ctypes.c_int]),
    "spx_set_option": (ctypes.c_int, [_i32, _i64]),
    "spx_get_option": (_i64, [_i32]),
    "spx_selftest_division": (ctypes.c_int, [_vp, _vp, _i64, _i64, ctypes.POINTER(ctypes.c_uint64),
                                             ctypes.POINTER(ctypes.c_double), _vp]),
    "spx_selftest_lazy_guard": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _vp, _vp,
                                               ctypes.POINTER(ctypes.c_uint64), _vp]),
    "spx_import_table": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp]),
    "spx_import_shard": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _i64, _vp]),
    "spx_export_table": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp]),
    "spx_init_state": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i64, _vp]),
    "spx_pick": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i64, _i32, _i32, _vp, _vp, _vp]),
    "spx_update": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_solve_workspace_bytes": (_i64, [_i32]),
    "spx_fused_workspace_bytes": (_i64, [_i32, _i32]),
    "spx_fused_pass": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _i32, _i32, _vp, _vp, _i64, _vp, _vp,
                                      _vp, _vp]),
    "spx_solve": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp,
                                 _i32, _i64, _i32, _vp, _i64, _pi32, _pi64, _vp]),
    "spx_extract": (ctypes.c_int, [_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "spx_solve_batched": (ctypes.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                         _vp, _vp, _vp]),
    "spx_batched_max_cells": (_i64, []),
    "spx_batched_fits": (_i32, [_i32, _i32]),
    "spx_batched_route": (_i32, [_i32, _i32, _i32]),
    "spx_solve_batched_cluster": (ctypes.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                                 _vp, _vp, _vp]),
    "spx_cluster_size": (_i32, [_i32, _i32]),
    "spx_solve_batched_global": (ctypes.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp,
                                                _vp, _vp, _vp]),
    "spx_global_min_cluster_size": (_i32, [_i32, _i32]),
    "spx_global_cluster_size": (_i32, [_i32, _i32, _i64]),
    "spx_ragged_plan_bytes": (_i64, [_i64]),
    "spx_ragged_plan": (ctypes.c_int, [_vp, _i64, _i32, _vp, _i64, _vp]),
    "spx_solve_batched_ragged": (ctypes.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_ragged_cluster_size": (_i32, [_vp, _i32]),
    "spx_sensitivity_batched": (ctypes.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_sensitivity_ragged": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_sensitivity_split": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _pi32,
                                             _vp]),
    "spx_warm_change_batched": (ctypes.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "spx_warm_change_ragged": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_warm_solve_batched": (ctypes.c_int, [_i32, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp,
                                              _vp, _vp, _vp, _vp, _vp]),
    "spx_warm_solve_ragged": (ctypes.c_int, [_vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "spx_shard_msg_doubles": (_i64, [_i32]),
    "spx_shard_candidate": (ctypes.c_int, [_vp, _vp, _i32, _i32, _i64, _i64, _i32, _i32, _vp, _vp, _vp]),
    "spx_shard_select": (ctypes.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _vp, ctypes.c_uint64, _vp]),
    "spx_shard_update": (ctypes.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _i64, _i64, _vp, _vp, _vp, _vp,
                                        _vp, _i32, _vp]),
    "spx_ahead_candidate": (ctypes.c_int, [_vp, _vp, _vp, _i32, _i32, _i64, _i64, _i32, _vp, _vp, _vp, _vp]),
    "spx_ahead_select": (ctypes.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _vp, _vp, ctypes.c_uint64, _vp]),
    "spx_device_alloc": (ctypes.c_int, [ctypes.POINTER(_vp), _i64]),
    "spx_device_free": (ctypes.c_int, [_vp]),
    "spx_ipc_handle_bytes": (ctypes.c_int, []),
    "spx_ipc_export": (ctypes.c_int, [_vp, _vp]),
    "spx_ipc_import": (ctypes.c_int, [_vp, ctypes.POINTER(_vp)]),
    "spx_ipc_close": (ctypes.c_int, [_vp]),
    "spx_mailbox_bytes": (_i64, [_i32, _i32]),
    "spx_peer_push": (ctypes.c_int, [_vp, _i32, _i32, _i32, _i32, ctypes.c_uint64, ctypes.POINTER(_vp), _vp]),
    "spx_shard_open": (ctypes.c_int, [ctypes.POINTER(_vp), _i32, _i32, _i32, _i32, _i64, _i64, _i32, _vp, _vp, _vp,
                                      _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "spx_shard_reset": (ctypes.c_int, [_vp]),
    "spx_shard_enqueue": (ctypes.c_int, [_vp, _i64, _vp]),
    "spx_shard_read": (ctypes.c_int, [_vp, _vp, _pi32, _vp]),
    "spx_shard_close": (ctypes.c_int, [_vp]),
    "spx_fshard_xbox_bytes": (_i64, [_i32, _i32]),
    "spx_fshard_open": (ctypes.c_int, [ctypes.POINTER(_vp), _i32, _i32, _i32, _i32, _i64, _i64, _i32, _vp, _vp, _vp, _vp,
                                       _vp, _vp, _i64, _vp, _vp, _vp, ctypes.POINTER(_vp)]),
    "spx_fshard_set_lookahead": (ctypes.c_int, [_vp, _i32]),
    "spx_fshard_enqueue": (ctypes.c_int, [_vp, _i64, _i32, _vp]),
    "spx_fshard_read": (ctypes.c_int, [_vp, _vp, _pi32, _vp]),
    "spx_fshard_close": (ctypes.c_int, [_vp]),
    "spx_fused_debug_stamps": (ctypes.c_int, [_vp, _i32, _i64, ctypes.POINTER(ctypes.c_uint64), _i32, _vp]),
    "spx_resident_debug": (ctypes.c_int, [ctypes.POINTER(ctypes.c_uint64)]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the library and bind every declared symbol (no GPU needed for this)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeUnavailable(
            f"{LIB_PATH} is missing: build it with `python -m simplex_method_solver_b200.build` "
            "(there is no CPU fallback)")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)           # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if L.spx_version() != ABI_VERSION:
        raise NativeUnavailable("libspx_b200.so ABI version mismatch")
    if L.spx_state_bytes() != ctypes.sizeof(SpxState):
        raise NativeUnavailable("spx_state layout mismatch between header and Python mirror")
    _lib = L
    return L


def lib() -> ctypes.CDLL:
    """The library, for compute calls: also requires a CUDA device."""
    import torch
    L = load()
    if not torch.cuda.is_available():
        raise NativeUnavailable("no CUDA device: the B200 pivot kernels cannot run (there is no CPU fallback)")
    return L


def call(name: str, *args) -> None:
    L = lib()
    rc = getattr(L, name)(*args)
    if rc != 0:
        raise SpxError(f"{name} failed ({rc}): {L.spx_last_error().decode(errors='replace')}")


def ptr(t) -> int:
    """Device/host pointer of a torch tensor (or None)."""
    return None if t is None else t.data_ptr()


def stream_handle() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
