"""ctypes binding of the C ABI in include/stratego_b200.h.

There is no CPU or pure-PyTorch fallback: if the shared library is missing or does not load,
importing the engine raises.
"""
import ctypes as C
import os

from . import _build

_i32, _i64, _u32, _u64, _vp = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_void_p

SX_ACTION_SPATIAL, SX_ACTION_1D = 0, 1
SX_AUTO_RESET, SX_SAMPLE_NEXT, SX_ALLOW_OSCILLATION, SX_RESET_RANDOM_SHUFFLE, SX_KERNEL_BASELINE = 1, 2, 4, 8, 16
SX_SAME_SETUP, SX_REPEAT_OTHER_SIDE = 32, 64
OBS_PO, OBS_FO, OBS_MASK = 1, 2, 4
SX_CHANNELS_EXTENDED, SX_CHANNELS_ORIGINAL = 0, 1
SX_DTYPE_F32, SX_DTYPE_BF16, SX_DTYPE_F16 = 0, 1, 2
SX_ALLOC_COMPRESSIBLE = 1
SX_KEY_STATE, SX_KEY_INFOSET = 0, 1
SX_LEAF_EVAL, SX_LEAF_OVER, SX_LEAF_STUCK = 0, 1, 2
SX_GUIDED_MAX_LEAVES = 1024


class SxConfigDesc(C.Structure):
    _fields_ = [("rows", _i32), ("cols", _i32), ("max_turns", _i32), ("usable_rows", _i32),
                ("piece_amounts", _i32 * 13), ("obstacles", _vp), ("captured_lut", _vp), ("recent_lut", _vp),
                ("unit_lut", _vp), ("p2_rot180", _i32), ("capture_capacity", _i32), ("obs_channel_mode", _i32),
                ("rank_lut", _vp), ("po_rank_lut", _vp), ("obs_dtype", _i32)]


class SxLayout(C.Structure):
    _fields_ = [(n, _i32) for n in ("rows", "cols", "cells", "spatial_channels", "spatial_actions", "action_size",
                                    "board_stride", "aux_stride", "captured_stride", "po_floats", "fo_floats",
                                    "setup_len", "pieces_per_side", "po_channels", "fo_channels",
                                    "obs_elem_bytes")]


class SxState(C.Structure):
    _fields_ = [("board", _vp), ("aux", _vp), ("captured", _vp)]


class SxOutputs(C.Structure):
    _fields_ = [(n, _vp) for n in ("partial_obs", "full_obs", "valid_mask", "reward", "done", "winner",
                                   "ending_invalid", "illegal", "player", "next_action", "terminal_partial_obs",
                                   "terminal_full_obs")]


class SxTree(C.Structure):
    _fields_ = [(n, _vp) for n in ("visits", "value", "parent", "first_child", "n_children", "action", "used")]


class SxGuidedTree(C.Structure):
    _fields_ = [(n, _vp) for n in ("visits", "value", "parent", "first_child", "n_children", "action", "prior", "used")]


class SxLaunchInfo(C.Structure):
    _fields_ = [(n, _i32) for n in ("warps_per_block", "blocks_per_sm", "smem_bytes_per_block", "num_sms",
                                    "grid_blocks", "regs_per_thread", "background_bytes", "thread_per_game")]


# every symbol include/stratego_b200.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "sx_last_error": (C.c_char_p, []),
    "sx_version": (C.c_int, []),
    "sx_config_create": (C.c_int, [C.POINTER(SxConfigDesc), C.POINTER(_vp)]),
    "sx_config_destroy": (None, [_vp]),
    "sx_config_layout": (C.c_int, [_vp, C.POINTER(SxLayout)]),
    "sx_config_set_tuning": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32]),
    "sx_config_set_start_states": (C.c_int, [_vp, SxState, _i64, _vp, _i64, _i64]),
    "sx_reset": (C.c_int, [_vp, SxState, _i64, _i64, _vp, _vp, _i32, _vp, _u64, _u32, _vp]),
    "sx_import_ref_state": (C.c_int, [_vp, SxState, _i64, _vp, _vp, _vp, _vp]),
    "sx_export_ref_state": (C.c_int, [_vp, SxState, _i64, _vp, _vp, _vp]),
    "sx_export_perspective_state": (C.c_int, [_vp, SxState, _i64, _vp, _vp, _vp]),
    "sx_valid_mask": (C.c_int, [_vp, SxState, _i64, _vp, _i32, _vp, _vp]),
    "sx_observe": (C.c_int, [_vp, SxState, _i64, _vp, SxOutputs, _vp]),
    "sx_step": (C.c_int, [_vp, SxState, _i64, _vp, _i32, _u32, SxOutputs, _vp]),
    "sx_step_all": (C.c_int, [_vp, SxState, _i64, _i64, _vp, _i32, _u32, _vp, _i32, _u64, SxOutputs, _vp, _vp]),
    "sx_sample_valid": (C.c_int, [_vp, _i64, _i32, _i64, _u64, _u32, _vp, _vp]),
    "sx_sample_logits": (C.c_int, [_vp, _i32, _vp, _i64, _i32, _i64, _u64, _u32, C.c_float, _vp, _vp, _vp]),
    "sx_sample_policy": (C.c_int, [_vp, SxState, _i64, _i64, _vp, _i32, _u64, _u32, C.c_float, _vp, _vp, _vp]),
    "sx_heuristic_rewards": (C.c_int, [_vp, SxState, _i64, _vp, _i32, _vp, _vp, _vp]),
    "sx_sample_hidden_states": (C.c_int, [_vp, SxState, _i64, _i64, _vp, _i32, _u64, _u32, SxState, _vp, _vp]),
    "sx_count_moves": (C.c_int, [_vp, SxState, _i64, _vp, _vp]),
    "sx_expand_moves": (C.c_int, [_vp, SxState, _i64, _vp, _i64, SxState, _vp, SxOutputs, _vp]),
    "sx_playout": (C.c_int, [_vp, SxState, _i64, _i64, _i32, _u64, _vp, SxOutputs, _vp]),
    "sx_state_keys": (C.c_int, [_vp, SxState, _i64, _vp, _u32, _vp, _vp]),
    "sx_search": (C.c_int, [_vp, SxState, _i64, _i64, _i32, _i32, _i32, C.c_float, _u64, SxTree, _vp]),
    "sx_guided_select": (C.c_int, [_vp, SxState, _i64, SxGuidedTree, _i32, C.c_float, C.c_float, SxState, _vp, _vp, _vp]),
    "sx_guided_backup": (C.c_int, [_vp, SxState, _i64, SxGuidedTree, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "sx_guided_select_many": (C.c_int, [_vp, SxState, _i64, SxGuidedTree, _i32, C.c_float, C.c_float, _i32, C.c_float,
                                        _vp, SxState, _vp, _vp, _vp]),
    "sx_guided_backup_many": (C.c_int, [_vp, SxState, _i64, SxGuidedTree, _i32, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "sx_step_all_launch_info": (C.c_int, [_vp, _u32, C.POINTER(SxLaunchInfo)]),
    "sx_device_alloc": (C.c_int, [_i32, _u64, _u32, C.POINTER(_vp), C.POINTER(_u32)]),
    "sx_device_free": (C.c_int, [_vp]),
    "sx_device_alloc_info": (C.c_int, [_vp, C.POINTER(_u64), C.POINTER(_u32), C.POINTER(_i64)]),
    "sx_host_env_create": (C.c_int, [_vp, _i64, _i64, _u32, _u32, _vp, _i32, _u64, _i32, C.POINTER(_vp)]),
    "sx_host_env_destroy": (None, [_vp]),
    "sx_host_env_reset": (C.c_int, [_vp, SxOutputs]),
    "sx_host_env_step": (C.c_int, [_vp, _vp, SxOutputs]),
    "sx_host_env_step_ex": (C.c_int, [_vp, _vp, _i32, _u32, SxOutputs]),
    "sx_host_env_step_device": (C.c_int, [_vp, _i32]),
    "sx_host_env_sync": (C.c_int, [_vp]),
    "sx_host_env_state": (C.c_int, [_vp, C.POINTER(SxState), C.POINTER(SxOutputs)]),
}

_lib = None


class StrategoB200Error(RuntimeError):
    pass


def library_path() -> str:
    return _build.LIB_PATH


def load(build_if_missing: bool = True):
    """Loads (building first when stale and nvcc is present) csrc/libstratego_b200.so."""
    global _lib
    if _lib is not None:
        return _lib
    # SX_LIB: load another build of the library instead, e.g. to time two builds against each other
    path = os.environ.get("SX_LIB") or _build.LIB_PATH
    if build_if_missing and path == _build.LIB_PATH and _build.is_stale():
        try:
            _build.build_extension()
        except Exception as exc:  # noqa: BLE001
            if not os.path.exists(path):
                raise StrategoB200Error(
                    "CUDA extension %s is missing and could not be built (%s). The B200 Stratego engine has no "
                    "CPU fallback." % (path, exc)) from exc
            # a library exists but is OLDER than its sources and the rebuild failed: running it would test code that
            # is not in the tree.  Allowed only where there is no compiler at all (a GPU box that received the prebuilt
            # library with fresh checkout timestamps); with nvcc present a failed build is an error.
            import shutil
            import warnings
            if shutil.which("nvcc") or os.path.exists("/usr/local/cuda/bin/nvcc"):
                raise StrategoB200Error("CUDA extension %s is stale and the rebuild failed: %s" % (path, exc)) from exc
            warnings.warn("stratego_env_b200: %s is older than its sources and could not be rebuilt (%s); using it "
                          "as is" % (path, exc), RuntimeWarning)
    if not os.path.exists(path):
        raise StrategoB200Error("CUDA extension %s is missing; run __graft_entry__.build(). There is no CPU "
                                "fallback." % path)
    lib = C.CDLL(path)
    for name, (restype, argtypes) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library out of sync
        fn.restype, fn.argtypes = restype, argtypes
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().sx_last_error()
        raise StrategoB200Error("%s failed: %s" % (what or "stratego_b200 call", msg.decode() if msg else rc))
