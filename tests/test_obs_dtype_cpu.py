"""No-GPU checks of the observation element type (sx_config_desc::obs_dtype): accepted values, the layout it reports,
the zero default, and the host layer's argument check."""
import ctypes

import numpy as np
import pytest
import torch


def _desc(keep):
    from stratego_env_b200 import _lib
    desc = _lib.SxConfigDesc()
    desc.rows, desc.cols, desc.max_turns, desc.usable_rows = 10, 10, 1000, 4
    for code, n in {1: 1, 2: 2, 3: 1, 9: 1, 10: 1, 11: 1, 12: 1}.items():
        desc.piece_amounts[code] = n
    keep += [np.zeros(100, np.uint8), np.zeros((12, 9), np.float32), np.zeros(5, np.float32), np.zeros(2, np.float32)]
    desc.obstacles, desc.captured_lut, desc.recent_lut, desc.unit_lut = (k.ctypes.data for k in keep[-4:])
    return desc


def _layout(lib, desc):
    from stratego_env_b200 import _lib
    handle = ctypes.c_void_p()
    assert lib.sx_config_create(ctypes.byref(desc), ctypes.byref(handle)) == 0, lib.sx_last_error()
    lay = _lib.SxLayout()
    assert lib.sx_config_layout(handle, ctypes.byref(lay)) == 0
    lib.sx_config_destroy(handle)
    return lay


@pytest.mark.parametrize("dtype,elem_bytes", [(0, 4), (1, 2), (2, 2)])
def test_obs_dtype_is_accepted_and_sets_the_element_size(dtype, elem_bytes):
    from stratego_env_b200 import _lib
    lib, keep = _lib.load(), []
    desc = _desc(keep)
    desc.obs_dtype = dtype
    lay = _layout(lib, desc)
    assert lay.obs_elem_bytes == elem_bytes
    # element counts keep their meaning whatever the element size
    assert (lay.po_floats, lay.fo_floats, lay.po_channels, lay.fo_channels) == (6700, 7900, 67, 79)


@pytest.mark.parametrize("dtype", [3, -1, 7])
def test_unknown_obs_dtype_is_rejected_by_name(dtype):
    from stratego_env_b200 import _lib
    lib, keep = _lib.load(), []
    desc = _desc(keep)
    desc.obs_dtype = dtype
    handle = ctypes.c_void_p()
    assert lib.sx_config_create(ctypes.byref(desc), ctypes.byref(handle)) != 0
    assert b"obs_dtype" in lib.sx_last_error()


def test_zeroed_descriptor_means_float32():
    from stratego_env_b200 import _lib
    lib, keep = _lib.load(), []
    desc = _desc(keep)
    assert desc.obs_dtype == 0 == _lib.SX_DTYPE_F32
    assert _layout(lib, desc).obs_elem_bytes == 4


@pytest.mark.parametrize("bad", [torch.int8, torch.float64, "bfloat16", None])
def test_bad_obs_dtype_is_a_value_error_before_any_device_is_needed(bad):
    from stratego_env_b200 import BatchedStrategoEnv, GameVersions
    from stratego_env_b200.config import MICRO_STRATEGO_CONFIG
    from stratego_env_b200.engine import StrategoEngine
    with pytest.raises(ValueError, match="obs_dtype"):
        BatchedStrategoEnv({"version": GameVersions.MICRO}, num_envs=4, obs_dtype=bad)
    with pytest.raises(ValueError, match="obs_dtype"):
        StrategoEngine(MICRO_STRATEGO_CONFIG, obs_dtype=bad)


def test_obs_dtype_codes_match_the_header():
    from stratego_env_b200 import _lib
    from stratego_env_b200.engine import obs_dtype_code
    assert [obs_dtype_code(t) for t in (torch.float32, torch.bfloat16, torch.float16)] == \
        [_lib.SX_DTYPE_F32, _lib.SX_DTYPE_BF16, _lib.SX_DTYPE_F16] == [0, 1, 2]
