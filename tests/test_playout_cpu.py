"""No-GPU checks of random playouts (sx_playout): the reference of tests/_playout_ref.py pinned to the unmodified
reference's recorded games of every variant, and the argument checks of the C ABI and of StrategoEngine.playout."""
import numpy as np
import pytest

from _expand_ref import logic
from _golden import VERSIONS, traj, unpack_mask
from _playout_ref import INVALID, OVER, TURN, WINNER, data, playout_ref
from _sampler_ref import step_words, uniform_valid_ref
from test_expand_moves_cpu import _config, _fake_state, _no_device_engine, _state

SEED = 0x1234_5678_9ABC_DEF0  # non-zero high word
GID0 = 3 << 32                 # gids above 2^32


@pytest.mark.parametrize("version", VERSIONS)
def test_one_ply_is_the_step_draw(version):
    """max_plies = 1 on every recorded state, both players to move: the move played is the step_words draw over the
    mask (the recorded one for the recorded player), an entry of that mask, and the successor is the oracle's step"""
    t = traj(version)
    orc = logic(version)
    R, C, A = int(t["rows"]), int(t["columns"]), int(t["channels"])
    states = t["states"].astype(np.int64)
    for flip in (False, True):
        for i in range(states.shape[0]):
            player = -int(t["players"][i]) if flip else int(t["players"][i])
            st = states[i]
            got, nxt, plies, _ = playout_ref(orc, st, player, GID0 + i, 0, SEED, 1)
            if data(st, OVER):
                assert plies == 0 and np.array_equal(got, st) and nxt == player, (version, flip, i)
                continue
            mask = orc.current_obs(st, player, obs_mode=0)[0].reshape(-1)
            if not flip:
                assert np.array_equal(mask != 0, unpack_mask(t["mask_bits"][i], R * C * A) != 0), (version, i)
            a = int(uniform_valid_ref(mask[None], step_words(np.array([GID0 + i]), data(st, TURN), 0, SEED))[0])
            assert mask[a] != 0, (version, flip, i)
            if a == A - 1:  # a stuck player: the noop is its only entry, and it loses by it
                assert mask.sum() == 1, (version, flip, i)
                want, want_player = orc.base_env.get_next_state(st, player, orc.base_env.action_size - 1)
                assert data(want, OVER) == 1 and data(want, WINNER) == -player, (version, flip, i)
            else:
                want, want_player = orc.apply_spatial_action(st, player, a)
            assert plies == 1 and np.array_equal(got, want) and nxt == want_player, (version, flip, i)


@pytest.mark.parametrize("version", VERSIONS)
def test_finished_states_play_nothing(version):
    """the recorded states of finished games play 0 plies and stay as they are, whatever the cap"""
    t = traj(version)
    orc = logic(version)
    states = t["states"].astype(np.int64)
    ended = [i for i in range(states.shape[0]) if data(states[i], OVER)]
    assert ended, version
    for i in ended:
        for cap in (0, 1, (1 << 31) - 1):
            got, nxt, plies, outcome = playout_ref(orc, states[i], t["players"][i], i, 0, SEED, cap)
            assert plies == 0 and np.array_equal(got, states[i]) and nxt == int(t["players"][i]), (version, i)
            assert outcome[0] == 1, (version, i)


@pytest.mark.parametrize("version", VERSIONS)
def test_playouts_compose(version):
    """ref(a) followed by ref(b) equals ref(a + b), on every fifth recorded state with both players to move"""
    t = traj(version)
    orc = logic(version)
    states = t["states"].astype(np.int64)
    for flip in (False, True):
        for i in range(0, states.shape[0], 5):
            player = -int(t["players"][i]) if flip else int(t["players"][i])
            whole = playout_ref(orc, states[i], player, GID0 + i, 7, SEED, 9)
            mid, mid_player, n1, _ = playout_ref(orc, states[i], player, GID0 + i, 7, SEED, 4)
            end, end_player, n2, outcome = playout_ref(orc, mid, mid_player, GID0 + i, 7, SEED, 5)
            assert np.array_equal(end, whole[0]) and end_player == whole[1], (version, flip, i)
            assert n1 + n2 == whole[2] and outcome == whole[3], (version, flip, i)


@pytest.mark.parametrize("version", VERSIONS)
def test_playouts_from_start_states_end(version):
    """from the recorded start states, each playout ends within max_turns plies, with a winner or an invalid ending by
    the turn limit, as the oracle's game-ended and invalid-result queries report"""
    t = traj(version)
    orc = logic(version)
    states = t["states"].astype(np.int64)
    starts = np.flatnonzero(t["game_start"])
    assert starts.size > 0, version
    for i in starts[:4]:
        max_turns = int(states[i][5][1, 0])
        got, player, plies, (over, winner, invalid) = playout_ref(orc, states[i], t["players"][i], GID0 + i, 0, SEED,
                                                                  (1 << 31) - 1)
        assert over == 1 and 0 < plies <= max_turns, (version, i, plies)
        assert bool(invalid) == orc.base_env.get_game_result_is_invalid(got), (version, i)
        ended = float(orc.base_env.get_game_ended(got, player))
        if invalid:
            assert winner == 0 and data(got, TURN) == max_turns and plies == max_turns, (version, i)
        else:
            assert winner in (1, -1) and ended == winner * player, (version, i)
        assert data(got, WINNER) == winner and data(got, INVALID) == invalid, (version, i)


# ---- argument checks without a device -------------------------------------------------------------------------------
def _playout_call(lib, cfg, st=None, num_envs=4, max_plies=5, scalars=None):
    from stratego_env_b200 import _lib
    return lib.sx_playout(cfg, _fake_state(0x10000) if st is None else st, num_envs, 0, max_plies, 1, 0x30000,
                          _lib.SxOutputs() if scalars is None else scalars, None)


@pytest.mark.parametrize("case,needle", [
    ("null config", b"null config"), ("null state", b"null state"), ("negative max_plies", b"max_plies"),
    *[("scalar " + n, b"must be null") for n in ("partial_obs", "full_obs", "valid_mask", "next_action",
                                                  "terminal_partial_obs", "terminal_full_obs")]])
def test_abi_refusals(case, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        kw = {"null state": dict(st=_lib.SxState()), "negative max_plies": dict(max_plies=-1)}.get(case, {})
        if case.startswith("scalar "):
            s = _lib.SxOutputs()
            setattr(s, case[len("scalar "):], 0x50000)
            kw = dict(scalars=s)
        assert _playout_call(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_no_games_is_a_no_op():
    """num_envs <= 0 launches nothing (fake pointers are never touched); the six scalar outputs and plies are
    accepted, and so is max_plies = 0 or INT32_MAX"""
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        scalars = _lib.SxOutputs()
        for i, n in enumerate(("reward", "done", "winner", "ending_invalid", "illegal", "player")):
            setattr(scalars, n, 0x60000 + 0x1000 * i)
        for n in (0, -3):
            for cap in (0, (1 << 31) - 1):
                assert _playout_call(lib, cfg, num_envs=n, max_plies=cap, scalars=scalars) == 0
    finally:
        lib.sx_config_destroy(cfg)


@pytest.mark.parametrize("state", [None, "state", (1, 2, 3), _state()], ids=["None", "str", "tuple", "host tensors"])
def test_engine_rejects_bad_state_before_touching_a_device(state, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="state"):
        eng.playout(state)


@pytest.mark.parametrize("max_plies", [-1, True, False, 1.0, 2.5, "7", 1 << 31, 1 << 40],
                         ids=["negative", "True", "False", "float", "fraction", "str", "2^31", "2^40"])
def test_engine_rejects_bad_max_plies_before_touching_a_device(max_plies, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="max_plies"):
        eng.playout(_state(), max_plies=max_plies)
