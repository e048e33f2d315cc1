"""No-GPU checks of move expansion (sx_count_moves / sx_expand_moves): the reference of tests/_expand_ref.py pinned to
the unmodified reference's recorded games of every variant, and the argument checks of the C ABI and of
StrategoEngine.expand_moves."""
import ctypes

import numpy as np
import pytest
import torch

from _expand_ref import action_list, expand_ref, logic
from _golden import VERSIONS, traj, transitions, unpack_mask


@pytest.mark.parametrize("version", VERSIONS)
def test_reference_contains_every_recorded_move_and_its_successor(version):
    """for every recorded transition states[i] -(actions_spatial[i])-> states[i+1]: the recorded action is in the
    reference's list, its child equals states[i+1] and the next player is the recorded one; the list is ascending"""
    t = traj(version)
    orc = logic(version)
    states = t["states"].astype(np.int64)
    for i in transitions(t):
        acts, kids, nxt = expand_ref(orc, states[i], t["players"][i])
        assert np.all(np.diff(acts) > 0), (version, i)
        j = np.flatnonzero(acts == int(t["actions_spatial"][i]))
        assert j.size == 1, (version, i)
        assert np.array_equal(kids[j[0]], states[i + 1]), (version, i)
        assert nxt[j[0]] == int(t["players"][i + 1]), (version, i)


@pytest.mark.parametrize("version", VERSIONS)
def test_reference_list_is_the_recorded_mask_without_the_noop(version):
    """on every recorded state the list equals the recorded mask entries outside the noop channel; the states a
    recorded game ended in have no children"""
    t = traj(version)
    orc = logic(version)
    R, C, A = int(t["rows"]), int(t["columns"]), int(t["channels"])
    states = t["states"].astype(np.int64)
    for i in range(states.shape[0]):
        flat = unpack_mask(t["mask_bits"][i], R * C * A)
        want = np.flatnonzero(flat)
        want = want[want % A != A - 1]
        assert np.array_equal(action_list(orc, states[i], t["players"][i]), want), (version, i)
    ended = [i + 1 for i in transitions(t) if t["dones"][i]]
    assert ended, version
    for i in ended:
        assert action_list(orc, states[i], t["players"][i]).size == 0, (version, i)


# ---- argument checks without a device -------------------------------------------------------------------------------
def _config():
    """a Barrage sx_config made without a device (sx_config_create needs none)"""
    from stratego_env_b200 import _lib
    from stratego_env_b200.config import (VERSION_CONFIGS, as_version, captured_lut, obstacle_map, piece_amounts_array,
                                          recent_moves_lut, unit_channel_lut)
    lib = _lib.load()
    cfg = VERSION_CONFIGS[as_version("barrage")]
    desc = _lib.SxConfigDesc()
    desc.rows, desc.cols, desc.max_turns, desc.usable_rows = 10, 10, 1000, 4
    for i, v in enumerate(piece_amounts_array(cfg["piece_amounts"])):
        desc.piece_amounts[i] = int(v)
    keep = [np.ascontiguousarray(obstacle_map(cfg).reshape(-1), dtype=np.uint8),
            np.ascontiguousarray(captured_lut(cfg["piece_amounts"]), dtype=np.float32),
            np.ascontiguousarray(recent_moves_lut(), dtype=np.float32),
            np.ascontiguousarray(unit_channel_lut(), dtype=np.float32)]
    desc.obstacles, desc.captured_lut, desc.recent_lut, desc.unit_lut = (a.ctypes.data for a in keep)
    handle = ctypes.c_void_p()
    _lib.check(lib.sx_config_create(ctypes.byref(desc), ctypes.byref(handle)), "sx_config_create")
    return lib, handle, keep


def _fake_state(base):
    from stratego_env_b200 import _lib
    return _lib.SxState(base, base + 0x1000, base + 0x2000)


OFFSETS, ACTIONS = 0x30000, 0x40000


def _expand_call(lib, cfg, st=None, out=None, offsets=OFFSETS, n_children=8, actions=ACTIONS, scalars=None):
    from stratego_env_b200 import _lib
    return lib.sx_expand_moves(cfg, _fake_state(0x10000) if st is None else st, 4, offsets, n_children,
                               _fake_state(0x20000) if out is None else out, actions,
                               _lib.SxOutputs() if scalars is None else scalars, None)


def _scalars_with(name):
    from stratego_env_b200 import _lib
    s = _lib.SxOutputs()
    setattr(s, name, 0x50000)
    return s


@pytest.mark.parametrize("case,needle", [
    ("null config", b"null config"), ("null state", b"null state"), ("null out", b"null out"),
    ("null actions", b"null actions"), ("null offsets", b"null offsets"), ("same board", b"out.board is st.board"),
    ("negative n_children", b"n_children"),
    *[("scalar " + n, b"must be null") for n in ("partial_obs", "full_obs", "valid_mask", "next_action",
                                                  "terminal_partial_obs", "terminal_full_obs")]])
def test_abi_refusals(case, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        st = _fake_state(0x10000)
        kw = {"null config": dict(), "null state": dict(st=_lib.SxState()), "null out": dict(out=_lib.SxState()),
              "null actions": dict(actions=None), "null offsets": dict(offsets=None), "same board": dict(out=st),
              "negative n_children": dict(n_children=-1)}.get(case)
        if case.startswith("scalar "):
            kw = dict(scalars=_scalars_with(case[len("scalar "):]))
        assert _expand_call(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_no_work_is_a_no_op():
    """num_envs <= 0 or n_children == 0 launches nothing (fake pointers are never touched), and the six scalar outputs
    are accepted"""
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        scalars = _lib.SxOutputs()
        for i, n in enumerate(("reward", "done", "winner", "ending_invalid", "illegal", "player")):
            setattr(scalars, n, 0x60000 + 0x1000 * i)
        assert _expand_call(lib, cfg, n_children=0, scalars=scalars) == 0
        assert lib.sx_expand_moves(cfg, _fake_state(0x10000), 0, OFFSETS, 8, _fake_state(0x20000), ACTIONS, scalars,
                                   None) == 0
        assert lib.sx_count_moves(cfg, _fake_state(0x10000), 0, 0x30000, None) == 0
        assert lib.sx_count_moves(cfg, _fake_state(0x10000), -5, 0x30000, None) == 0
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_count_refusals():
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        assert lib.sx_count_moves(None, _fake_state(0x10000), 4, 0x30000, None) != 0
        assert b"null config" in lib.sx_last_error()
        assert lib.sx_count_moves(cfg, _lib.SxState(), 4, 0x30000, None) != 0
        assert b"null state" in lib.sx_last_error()
        assert lib.sx_count_moves(cfg, _fake_state(0x10000), 4, None, None) != 0
        assert b"null counts" in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def _no_device_engine(monkeypatch):
    """a Barrage StrategoEngine shell whose every library call or device query fails the test"""
    from stratego_env_b200 import _lib, engine

    def touched(*a, **k):
        raise AssertionError("the device or the library was reached before the argument check")
    eng = engine.StrategoEngine.__new__(engine.StrategoEngine)
    eng.lib = type("NoLib", (), {"__getattr__": lambda self, name: touched})()
    eng.device = torch.device("cuda", 0)
    lay = _lib.SxLayout()
    lay.board_stride, lay.aux_stride, lay.captured_stride = 112, 8, 16
    eng.layout = lay
    for name in ("is_available", "current_stream", "current_device", "synchronize"):
        monkeypatch.setattr(torch.cuda, name, touched)
    return eng


def _state(B=4):
    from stratego_env_b200.engine import DeviceState
    return DeviceState(torch.zeros(B, 112, dtype=torch.uint8), torch.zeros(B, 8, dtype=torch.int16),
                       torch.zeros(B, 16, dtype=torch.int16))


@pytest.mark.parametrize("state", [None, "state", (1, 2, 3), _state()], ids=["None", "str", "tuple", "host tensors"])
def test_engine_rejects_bad_state_before_touching_a_device(state, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="state"):
        eng.expand_moves(state)

