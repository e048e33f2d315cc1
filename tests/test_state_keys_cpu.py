"""No-GPU checks of position keys (sx_state_keys): the reference of tests/_keys_ref.py on the recorded games of every
variant (keys equal exactly where the positions are, information-set keys blind to determinization and sensitive to
everything else), its pinned values, and the argument checks of the C ABI and of StrategoEngine.state_keys."""
import numpy as np
import pytest
import torch

from _golden import TRAJ_LABELS, VERSIONS, traj
from _hidden_ref import hidden_cells, sample_hidden_ref
from _keys_ref import state_keys_ref, zobrist
from test_expand_moves_cpu import _config, _fake_state, _no_device_engine, _state

TURN = (5, 0, 0)


def _both_players(t):
    """every recorded state twice: with the recorded player to move and with the other one"""
    states = t["states"].astype(np.int64)
    players = t["players"].astype(np.int64)
    return np.concatenate([states, states]), np.concatenate([players, -players])


def _what_the_mover_knows(dense, player):
    """the states with the true rank of every piece hidden from the player to move replaced by UNKNOWN (13)"""
    hidden, _, opp, _ = hidden_cells(dense, player, None)
    out = dense.reshape(dense.shape[0], dense.shape[1], -1).copy()
    rows = np.arange(dense.shape[0])
    out[rows, opp] = np.where(hidden, 13, out[rows, opp])
    return out.reshape(dense.shape)


def _classes(rows):
    return np.unique(np.array(rows, dtype=object), return_inverse=True)[1]


@pytest.mark.parametrize("info", [False, True], ids=["state", "infoset"])
def test_keys_equal_exactly_where_the_positions_are_equal(info):
    """over every recorded state of every trajectory (all 11 variants), each with both players to move: equal keys
    exactly for equal (board size, state, player) -- for the information-set key of the player to move, for equal
    (board size, state with the pieces hidden from that player as UNKNOWN, player) -- and no collision otherwise"""
    ident, keys = [], []
    for label in TRAJ_LABELS:
        dense, player = _both_players(traj(label))
        shape = np.array(dense.shape[2:], dtype=np.int64)
        seen = _what_the_mover_knows(dense, player) if info else dense
        ident += [shape.tobytes() + d.tobytes() + p.tobytes() for d, p in zip(seen, player)]
        keys.append(state_keys_ref(dense, player, info_set=info, viewer=None))
    pos, kid = _classes(ident), _classes(np.concatenate(keys))
    assert pos.max() + 1 < len(ident)  # the recordings do hold repeated positions
    # a bijection between position classes and key classes
    assert np.unique(np.stack([pos, kid]), axis=1).shape[1] == pos.max() + 1 == kid.max() + 1


@pytest.mark.parametrize("version", VERSIONS)
def test_state_key_and_both_information_set_keys_differ(version):
    dense, player = _both_players(traj(version))
    B = dense.shape[0]
    s = state_keys_ref(dense, player)
    plus = state_keys_ref(dense, player, info_set=True, viewer=np.ones(B))
    minus = state_keys_ref(dense, player, info_set=True, viewer=-np.ones(B))
    assert np.all(s != plus) and np.all(s != minus) and np.all(plus != minus)
    mover = state_keys_ref(dense, player, info_set=True)
    assert np.array_equal(mover, np.where(player == 1, plus, minus))
    # anything but 1 is player -1
    assert np.array_equal(state_keys_ref(dense, player, info_set=True, viewer=np.full(B, 7)), minus)


@pytest.mark.parametrize("version", VERSIONS)
@pytest.mark.parametrize("viewer", [1, -1, None], ids=["plus", "minus", "mover"])
def test_information_set_keys_are_blind_to_determinization(version, viewer):
    """every world _hidden_ref draws for a viewer has its source's information-set key for that viewer; its state key
    differs exactly where the world's ranks differ from the source's"""
    dense, player = _both_players(traj(version))
    B = dense.shape[0]
    view = None if viewer is None else np.full(B, viewer)
    K = 8
    worlds, status = sample_hidden_ref(dense, player, view, K, seed=0xC0FFEE_0000_0001, draw=3)
    ok = np.repeat(status == 0, K)
    wp = np.repeat(player, K)
    wv = None if view is None else np.repeat(view, K)
    src = np.repeat(state_keys_ref(dense, player, info_set=True, viewer=view), K)
    assert np.array_equal(state_keys_ref(worlds, wp, info_set=True, viewer=wv), src)
    same = (worlds.reshape(B * K, -1) == np.repeat(dense, K, axis=0).reshape(B * K, -1)).all(1)
    moved = state_keys_ref(worlds, wp) != np.repeat(state_keys_ref(dense, player), K)
    assert np.array_equal(moved, ~same)
    assert moved[ok].any()  # some worlds do differ


def _midgame(version="barrage"):
    """a recorded state with a revealed piece, a piece that has moved, both recent-move records and a capture"""
    t = traj(version)
    for i, st in enumerate(t["states"].astype(np.int64)):
        revealed = (st[0] != 0) & (st[3] == st[0])
        if revealed.any() and (st[6] != 0).any() and (st[7] != 0).any() and st[8:32].any() and \
                ((st[0] != 0) & (st[32] == 0)).any():
            return st, int(t["players"][i])
    raise AssertionError("no such state recorded")


def _edits(st):
    """(name, edited copy) for each kind of change the keys must see"""
    out = []
    e = st.copy()
    r, c = np.argwhere((st[0] != 0) & (st[3] == st[0]))[0]
    e[0, r, c] = e[3, r, c] = 1 if st[0, r, c] != 1 else 2
    out.append(("revealed rank", e))
    e = st.copy()
    r, c = np.argwhere(st[0] != 0)[0]
    e[32, r, c] ^= 1
    out.append(("still bit", e))
    e = st.copy()
    r, c = np.argwhere(st[6] < 0)[0]
    e[6, r, c] = -3 if st[6, r, c] != -3 else -1
    out.append(("recent move code", e))
    e = st.copy()
    e[6][st[6] == 1] = 0
    r, c = np.argwhere(st[6] == 0)[0]
    e[6, r, c] = 1
    out.append(("recent move square", e))
    e = st.copy()
    layer, r, c = np.argwhere(st[8:32] != 0)[0]
    e[8 + layer, r, c] += 1
    out.append(("captured counter", e))
    e = st.copy()
    e[TURN] += 1
    out.append(("turn", e))
    return out


@pytest.mark.parametrize("info", [False, True], ids=["state", "infoset"])
def test_keys_see_every_public_change(info):
    """a revealed rank, a still bit, a recent-move entry, a captured counter, the turn and the player to move each
    change the key (for the information-set key: of either viewer)"""
    st, player = _midgame()
    for viewer in ((None,) if not info else (1, -1)):
        view = None if viewer is None else np.array([viewer])
        base = state_keys_ref(st[None], [player], info_set=info, viewer=view)[0]
        for name, e in _edits(st):
            assert not np.array_equal(e, st), name
            assert state_keys_ref(e[None], [player], info_set=info, viewer=view)[0] != base, (name, viewer)
        assert state_keys_ref(st[None], [-player], info_set=info, viewer=view)[0] != base, ("player", viewer)


def test_information_set_key_ignores_hidden_ranks_only():
    """changing the true rank of an unrevealed piece leaves the information-set key of its owner's opponent alone and
    changes its owner's and the state key, for pieces of either player"""
    st, player = _midgame()
    keys = lambda s, v: state_keys_ref(s[None], [player], info_set=v is not None,  # noqa: E731
                                       viewer=None if v is None else np.array([v]))[0]
    for owner, opponent in ((0, -1), (1, 1)):
        hidden, _, _, _ = hidden_cells(st[None], [player], np.array([opponent]))
        cells = np.flatnonzero(hidden[0])
        assert cells.size, owner
        r, c = divmod(int(cells[0]), st.shape[2])
        e = st.copy()
        e[owner, r, c] = 1 if st[owner, r, c] != 1 else 2
        assert keys(e, opponent) == keys(st, opponent), owner
        assert keys(e, -opponent) != keys(st, -opponent) and keys(e, None) != keys(st, None), owner


def test_obstacle_layer_is_not_keyed():
    st, player = _midgame()
    e = st.copy()
    e[2] = 1 - e[2]
    e[2][(st[0] != 0) | (st[1] != 0)] = 0
    assert state_keys_ref(e[None], [player])[0] == state_keys_ref(st[None], [player])[0]


def test_pinned_values():
    """the construction is fixed: tables kept across processes and versions stay valid"""
    assert int(zobrist(0, 34, 1)) == 0xEF45835C4E951D1D
    assert int(zobrist(17, 5, -1)) == 0x6510BC4E9DAA0E31
    t = traj("barrage")
    assert int(state_keys_ref(t["states"][:1].astype(np.int64), t["players"][:1])[0]) == 0x1534E3058FDB4729


# ---- argument checks without a device -------------------------------------------------------------------------------
KEYS, VIEWER = 0x30000, 0x40000


@pytest.mark.parametrize("case,needle", [
    ("null config", b"null config"), ("null state", b"null state"), ("null keys", b"null keys"),
    ("mode 2", b"unknown mode"), ("mode 2^31", b"unknown mode"), ("viewer in state mode", b"viewer_d must be NULL")])
def test_abi_refusals(case, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        args = dict(cfg=cfg, st=_fake_state(0x10000), viewer=None, mode=_lib.SX_KEY_STATE, keys=KEYS)
        args.update({"null config": dict(cfg=None), "null state": dict(st=_lib.SxState()), "null keys": dict(keys=None),
                     "mode 2": dict(mode=2), "mode 2^31": dict(mode=1 << 31),
                     "viewer in state mode": dict(viewer=VIEWER)}[case])
        assert lib.sx_state_keys(args["cfg"], args["st"], 4, args["viewer"], args["mode"], args["keys"], None) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_no_games_is_a_no_op():
    """num_envs <= 0 launches nothing (fake pointers are never touched), in both modes, with and without a viewer"""
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        for n in (0, -3):
            assert lib.sx_state_keys(cfg, _fake_state(0x10000), n, None, _lib.SX_KEY_STATE, KEYS, None) == 0
            for viewer in (None, VIEWER):
                assert lib.sx_state_keys(cfg, _fake_state(0x10000), n, viewer, _lib.SX_KEY_INFOSET, KEYS, None) == 0
    finally:
        lib.sx_config_destroy(cfg)


@pytest.mark.parametrize("state", [None, "state", (1, 2, 3), _state()], ids=["None", "str", "tuple", "host tensors"])
def test_engine_rejects_bad_state_before_touching_a_device(state, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="state"):
        eng.state_keys(state)


def _device_state(B=4):
    """a state of meta tensors on the engine's device: passes the host checks and cannot be touched"""
    from stratego_env_b200.engine import DeviceState
    st = _state(B)
    return DeviceState(*(torch.empty_like(t, device="meta") for t in (st.board, st.aux, st.captured)))


@pytest.mark.parametrize("kw,needle", [
    (dict(viewer=torch.ones(4, dtype=torch.int8)), "info_set=True"),
    (dict(info_set=1), "info_set"), (dict(info_set="yes"), "info_set"),
    (dict(info_set=True, viewer=torch.ones(3, dtype=torch.int8)), "viewer"),
    (dict(info_set=True, viewer=torch.ones(4, dtype=torch.float32)), "viewer"),
    (dict(info_set=True, viewer=torch.ones(4, dtype=torch.bool)), "viewer"),
    (dict(info_set=True, viewer=[1, 1, 1, 1]), "viewer"),
    (dict(info_set=True, viewer=np.ones(4, dtype=np.int8)), "viewer")],
    ids=["viewer without info_set", "info_set int", "info_set str", "short viewer", "float viewer", "bool viewer",
         "list viewer", "numpy viewer"])
def test_engine_rejects_bad_arguments_before_touching_a_device(kw, needle, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    eng.device = torch.device("meta")
    with pytest.raises(ValueError, match=needle):
        eng.state_keys(_device_state(), **kw)
