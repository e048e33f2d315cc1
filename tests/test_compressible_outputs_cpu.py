"""No-GPU checks of the library's device allocator (sx_device_alloc / sx_device_free / sx_device_alloc_info) and of
StrategoEngine's ``compressible_outputs`` argument: exported symbols, flag and argument validation."""
import ctypes

import pytest
import torch


def test_allocator_symbols_are_exported():
    from stratego_env_b200 import _lib
    raw = ctypes.CDLL(_lib.library_path())
    for name in ("sx_device_alloc", "sx_device_free", "sx_device_alloc_info"):
        assert hasattr(raw, name) and name in _lib.SYMBOLS
    assert _lib.SX_ALLOC_COMPRESSIBLE == 1


@pytest.mark.parametrize("flags", [2, 0x80000000, 0xFFFFFFFF, 3])
def test_unknown_flag_bits_are_rejected(flags):
    from stratego_env_b200 import _lib
    lib = _lib.load()
    ptr, granted = ctypes.c_void_p(123), ctypes.c_uint32(7)
    assert lib.sx_device_alloc(0, 1 << 20, flags, ctypes.byref(ptr), ctypes.byref(granted)) != 0
    assert b"unknown flags" in lib.sx_last_error()
    assert ptr.value is None and granted.value == 0  # outputs cleared on failure


def test_null_out_pointer_is_rejected():
    from stratego_env_b200 import _lib
    lib = _lib.load()
    assert lib.sx_device_alloc(0, 1 << 20, _lib.SX_ALLOC_COMPRESSIBLE, None, None) != 0
    assert b"null ptr" in lib.sx_last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
@pytest.mark.parametrize("device", [0, -1, 1 << 20])
def test_allocation_without_a_device_fails_cleanly(device):
    from stratego_env_b200 import _lib
    lib = _lib.load()
    ptr = ctypes.c_void_p()
    assert lib.sx_device_alloc(device, 4096, _lib.SX_ALLOC_COMPRESSIBLE, ctypes.byref(ptr), None) != 0
    assert b"no CUDA device" in lib.sx_last_error()
    assert ptr.value is None


def test_negative_device_is_rejected():
    from stratego_env_b200 import _lib
    lib = _lib.load()
    ptr = ctypes.c_void_p()
    assert lib.sx_device_alloc(-1, 4096, 0, ctypes.byref(ptr), None) != 0
    assert b"no CUDA device -1" in lib.sx_last_error()


def test_free_accepts_null_and_refuses_foreign_pointers():
    from stratego_env_b200 import _lib
    lib = _lib.load()
    assert lib.sx_device_free(None) == 0
    assert lib.sx_device_free(ctypes.c_void_p(0x1000)) != 0
    assert b"not allocated by sx_device_alloc" in lib.sx_last_error()


def test_alloc_info_counts_and_refuses_foreign_pointers():
    from stratego_env_b200 import _lib
    lib = _lib.load()
    live = ctypes.c_int64(-1)
    assert lib.sx_device_alloc_info(None, None, None, ctypes.byref(live)) == 0
    assert live.value >= 0
    assert lib.sx_device_alloc_info(ctypes.c_void_p(0x1000), None, None, None) != 0


@pytest.mark.parametrize("value", [1, 0, "yes", "auto", 1.0, [True]])
def test_engine_rejects_a_bad_compressible_outputs_value_before_touching_a_device(value, monkeypatch):
    from stratego_env_b200 import engine
    from stratego_env_b200.config import VERSION_CONFIGS, as_version

    def no_device(*a, **k):
        raise AssertionError("the device was queried before the argument check")
    monkeypatch.setattr(torch.cuda, "is_available", no_device)
    with pytest.raises(ValueError, match="compressible_outputs"):
        engine.StrategoEngine(VERSION_CONFIGS[as_version("barrage")], compressible_outputs=value)


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the behaviour without a CUDA device")
@pytest.mark.parametrize("value", [None, True, False])
def test_engine_accepts_the_valid_values_and_still_needs_a_device(value):
    from stratego_env_b200 import _lib, engine
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    with pytest.raises(_lib.StrategoB200Error, match="needs a CUDA device"):
        engine.StrategoEngine(VERSION_CONFIGS[as_version("barrage")], compressible_outputs=value)
