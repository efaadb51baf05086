"""ctypes binding of include/caro_b200.h (the drop-in boundary).  No torch types cross it: device
buffers are passed as raw pointers (``tensor.data_ptr()``), streams as ``cudaStream_t`` integers."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcaro_b200.so")

GAME_CONNECT4, GAME_MNK, GAME_CARO = 0, 1, 2


class CaroError(RuntimeError):
    pass


class EngineConfig(C.Structure):
    _fields_ = [("game", C.c_int32), ("n", C.c_int32), ("k", C.c_int32), ("games", C.c_int32),
                ("trees_per_game", C.c_int32), ("max_batch", C.c_int32), ("node_capacity", C.c_int32),
                ("replay_capacity", C.c_int32), ("c_puct", C.c_double), ("alpha", C.c_double),
                ("explore", C.c_double), ("seed", C.c_uint64), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


FLAG_VIRTUAL_LOSS, FLAG_MASK_PRIORS, FLAG_FRESH_TREE, FLAG_RECYCLE_TREE, FLAG_COMPACT_TREE = 1, 2, 4, 8, 16


_P = C.c_void_p
_SIGNATURES = {
    "caro_abi_version": (C.c_int, []),
    "caro_last_error": (C.c_char_p, []),
    "caro_device_count": (C.c_int, []),
    "caro_boards_apply": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "caro_boards_legal_mask": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_int64, _P, _P]),
    "caro_boards_encode_planes": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, _P, C.c_int64, _P, _P]),
    "caro_backup_path": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_float, _P]),
    "caro_net_blob_floats": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "caro_net_blob_floats_deep": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "caro_net_blob_floats_shape": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "caro_net_create": (C.c_int, [C.c_int, C.c_int, C.c_int, _P, C.c_size_t, C.POINTER(_P)]),
    "caro_net_create_shape": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_size_t, C.POINTER(_P)]),
    "caro_net_update": (C.c_int, [_P, _P, C.c_size_t]),
    "caro_net_destroy": (None, [_P]),
    "caro_net_set_trace": (C.c_int, [_P, _P]),
    "caro_net_set_grid_limit": (C.c_int, [_P, C.c_int]),
    "caro_net_forward": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int64, _P, _P, C.c_int, _P]),
    "caro_engine_workspace_bytes": (C.c_size_t, [C.POINTER(EngineConfig)]),
    "caro_engine_create": (C.c_int, [C.POINTER(EngineConfig), _P, C.c_size_t, C.POINTER(_P), _P]),
    "caro_engine_destroy": (None, [_P]),
    "caro_engine_region": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                     C.POINTER(C.c_int32), C.POINTER(C.c_int64 * 4)]),
    "caro_engine_reset": (C.c_int, [_P, _P, C.c_int, _P]),
    "caro_engine_set_roots": (C.c_int, [_P, _P, _P, _P]),
    "caro_engine_select": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P]),
    "caro_engine_plan": (C.c_int, [_P, C.c_int, _P]),
    "caro_engine_expand_backup": (C.c_int, [_P, C.c_int, _P, _P, _P]),
    "caro_engine_search": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "caro_engine_root_policy": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, _P, _P]),
    "caro_engine_advance": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, _P, _P]),
    "caro_engine_play": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "caro_engine_profile": (C.c_int, [_P, C.c_int]),
    "caro_engine_profile_read": (C.c_int, [_P, C.POINTER(C.c_double * 5), C.POINTER(C.c_uint64), _P]),
    "caro_engine_play_multi": (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    "caro_engine_replay_gather": (C.c_int, [_P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "caro_engine_counters": (C.c_int, [_P, C.POINTER(C.c_uint64 * 8), _P]),
    "caro_engine_set_resign": (C.c_int, [_P, C.c_int, C.c_double, C.c_double, _P]),
    "caro_engine_set_solver": (C.c_int, [_P, C.c_int, _P]),
    "caro_engine_set_gumbel": (C.c_int, [_P, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, _P]),
    "caro_engine_gumbel_plan": (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
}

_lib = None


def exported_symbols():
    return sorted(_SIGNATURES)


def lib():
    """Loads the CUDA library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CaroError("%s is missing: run `python __graft_entry__.py` (build()) first; "
                            "there is no CPU fallback" % LIB_PATH)
        # CARO_B200_LIB: developer switch for A/B runs of two builds on the same GPU box (tools/ only)
        handle = C.CDLL(os.environ.get("CARO_B200_LIB") or LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.caro_abi_version() != 2:
            raise CaroError("libcaro_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        raise CaroError("libcaro_b200 error %d: %s" % (rc, lib().caro_last_error().decode()))


def require_cuda():
    if lib().caro_device_count() <= 0:
        raise CaroError("no CUDA device visible: caro_ai_b200 has no CPU fallback")
