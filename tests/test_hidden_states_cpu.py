"""No-GPU checks of hidden-piece sampling (sx_sample_hidden_states): the numpy reference (tests/_hidden_ref.py) against
the contract on the recorded states of every variant, exact uniformity, draw independence, and the argument checks of
the C ABI and of StrategoEngine.sample_hidden_states.

The contract: the hidden cells are the cells of the viewer's opponent whose piece is not revealed; a sample places the
multiset of their true codes on them uniformly at random among the placements that put no flag or bomb on a cell whose
piece has moved.  Nothing the viewer sees may change: its partial observation and its valid-action mask equal the
original's byte for byte."""
import ctypes
import itertools

import numpy as np
import pytest
import scipy.stats
import torch

from _golden import VERSIONS, custom_toys, traj
from _hidden_ref import BOMB, FLAG, code_counts, hidden_cells, inferred_multiset, sample_hidden_ref

P_MIN = 1e-5  # chi-square p-value threshold; every draw below is at a fixed seed, so a pass is reproducible


def _cfg(version):
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    return VERSION_CONFIGS[as_version(version)]


def _amounts(cfg):
    from stratego_env_b200.config import piece_amounts_array
    return piece_amounts_array(cfg["piece_amounts"])


def _states(version, stride=1):
    t = traj(version)
    return t["states"][::stride].astype(np.int64), t["players"][::stride].astype(np.int64)


# ---- the contract on every recorded state --------------------------------------------------------------------------
@pytest.mark.parametrize("viewer", [1, -1, None])
@pytest.mark.parametrize("version", VERSIONS)
def test_samples_keep_everything_the_viewer_knows(version, viewer):
    """on every recorded state: only true ranks of the opponent's unrevealed pieces change, the hidden multiset is kept
    and equals piece_amounts - captured - revealed alive, no flag or bomb sits on a moved cell"""
    states, players = _states(version)
    B, K = states.shape[0], 3
    vw = None if viewer is None else np.full(B, viewer)
    samples, status = sample_hidden_ref(states, players, vw, K, seed=0x1234_5678_9ABC, draw=7, env_base=3)
    assert not status.any()
    hidden, still, opp, true = hidden_cells(states, players, vw)
    cnt = code_counts(hidden, true)
    assert np.array_equal(cnt, inferred_multiset(states, players, vw, _amounts(_cfg(version))))
    R, C = states.shape[2:]
    orig = np.repeat(states, K, axis=0).reshape(B * K, 34, R * C)
    got = samples.reshape(B * K, 34, R * C)
    rows = np.arange(B * K)
    hid_k, still_k, opp_k = np.repeat(hidden, K, 0), np.repeat(still, K, 0), np.repeat(opp, K)
    # every layer but the opponent's true ranks is untouched, and those only on hidden cells
    changed = got != orig
    changed[rows, opp_k] &= ~hid_k
    assert not changed.any()
    new_true = got[rows, opp_k]
    assert ((new_true != 0) == hid_k | (orig[rows, opp_k] != 0)).all()
    assert np.array_equal(code_counts(hid_k, new_true), np.repeat(cnt, K, 0))
    immovable = (new_true == FLAG) | (new_true == BOMB)
    assert not (hid_k & immovable & ~still_k).any()
    # the samples do differ from the truth somewhere (the draw is not the identity)
    if hidden.sum(1).max() > 1:
        assert (new_true != orig[rows, opp_k]).any()


@pytest.mark.parametrize("mode", ["extended", "original"])
@pytest.mark.parametrize("version", VERSIONS)
def test_viewer_observation_and_mask_are_unchanged(version, mode):
    """the viewer's partial observation (both channel modes) and spatial mask of every sample equal the original's"""
    from oracle.binding import OracleEnvLogic
    cfg = _cfg(version)
    orc = OracleEnvLogic(cfg["rows"], cfg["columns"], cfg["piece_amounts"], obs_channel_mode=mode)
    states, players = _states(version, stride=3)
    B, K = states.shape[0], 2
    for viewer in (1, -1):
        vw = np.full(B, viewer)
        samples, _ = sample_hidden_ref(states, players, vw, K, seed=99, draw=viewer & 0xFFFFFFFF)
        for b in range(B):
            m0, po0, _ = orc.current_obs(states[b], viewer, 1)
            for k in range(K):
                m1, po1, _ = orc.current_obs(samples[b * K + k], viewer, 1)
                assert np.array_equal(m0, m1), (version, b, k)
                assert np.array_equal(po0.view(np.uint32), po1.view(np.uint32)), (version, b, k)


@pytest.mark.parametrize("version", VERSIONS)
def test_oracle_plays_on_from_samples(version):
    """random legal play (a few dozen plies) from sampled states runs through the oracle without error"""
    from oracle.binding import OracleEnvLogic
    cfg = _cfg(version)
    orc = OracleEnvLogic(cfg["rows"], cfg["columns"], cfg["piece_amounts"])
    env = orc.base_env
    states, players = _states(version, stride=max(1, len(traj(version)["states"]) // 24))
    samples, _ = sample_hidden_ref(states, players, None, 2, seed=5)
    rng = np.random.default_rng(len(version))
    plies = 0
    for i in range(samples.shape[0]):
        s, p = samples[i], int(players[i // 2])
        for _ in range(40):
            if env.get_game_ended(s, p) != 0:
                break
            mask, _, _ = orc.current_obs(s, p, 0)
            valid = np.flatnonzero(mask.reshape(-1))
            s, p = orc.apply_spatial_action(s, p, int(rng.choice(valid)))
            plies += 1
    assert plies > 0


# ---- exact uniformity ---------------------------------------------------------------------------------------------
def _placements(codes, still):
    """every distinct assignment of the multiset `codes` to the cells, no flag / bomb on a non-still cell"""
    out = set()
    for perm in itertools.permutations(codes):
        if all(still[i] or perm[i] < FLAG for i in range(len(perm))):
            out.add(perm)
    return sorted(out)


def _chi2_over_placements(state, player, viewer, n=200_000, seed=2024):
    states, players = state[None], np.asarray([player])
    vw = np.asarray([viewer])
    hidden, still, _, true = hidden_cells(states, players, vw)
    cells = np.flatnonzero(hidden[0])
    places = _placements(tuple(true[0, cells]), still[0, cells])
    assert len(places) >= 2
    samples, status = sample_hidden_ref(states, players, vw, n, seed=seed, draw=1)
    assert not status.any()
    opp = 1 if viewer == 1 else 0
    got = samples.reshape(n, 34, -1)[:, opp][:, cells]
    index = {p: j for j, p in enumerate(places)}
    keys = [tuple(r) for r in got]
    assert all(k in index for k in keys)  # only consistent placements are drawn
    counts = np.bincount([index[k] for k in keys], minlength=len(places))
    p = scipy.stats.chisquare(counts).pvalue
    assert p > P_MIN, (len(places), p)
    assert counts.min() > 0
    return len(places)


def _pick(states, players, viewer, lo=6, hi=2000):
    """the recorded state with the most consistent placements within [lo, hi] and, if any, a moved hidden piece"""
    best, best_key = None, None
    for i in range(len(states)):
        h, s, _, t = hidden_cells(states[i:i + 1], players[i:i + 1], np.asarray([viewer]))
        cells = np.flatnonzero(h[0])
        if not 2 <= cells.size <= 8:
            continue
        n = len(_placements(tuple(t[0, cells]), s[0, cells]))
        key = (bool((~s[0, cells]).any()), n)
        if lo <= n <= hi and (best_key is None or key > best_key):
            best, best_key = i, key
    return best


@pytest.mark.parametrize("version,viewer", [("micro", 1), ("micro", -1), ("tiny", 1), ("tiny", -1)])
def test_uniform_over_every_placement_stock_toys(version, viewer):
    states, players = _states(version)
    i = _pick(states, players, viewer, lo=2)
    assert i is not None
    _chi2_over_placements(states[i], players[i], viewer)


def test_uniform_over_every_placement_custom_toy():
    """8 pieces a side on 4x4 (flag, two bombs, three scouts): a mid-game state with moved hidden pieces"""
    g = custom_toys()
    states = g["toy_eight_pieces_4x4_states"].astype(np.int64)
    players = g["toy_eight_pieces_4x4_players"].astype(np.int64)
    i = _pick(states, players, 1)
    assert i is not None
    assert _chi2_over_placements(states[i], players[i], 1) >= 6


def test_uniform_over_every_placement_hand_built_barrage():
    """a Barrage start position with the general and marshal revealed and a scout and the miner moved: flag and bomb
    on 2 of the 4 still cells (12 ways) times spy, scout, scout, miner on the rest (12 ways) = 144 placements"""
    t = traj("barrage")
    s = t["states"][0].astype(np.int64).copy()
    viewer, opp = 1, 1
    true, po, still = s[opp], s[3 + opp], s[32 + opp]
    for code in (9, 10):  # general, marshal: revealed
        r, c = np.argwhere(true == code)[0]
        po[r, c] = code
    for code in (2, 3):   # one scout and the miner have moved
        r, c = np.argwhere(true == code)[0]
        still[r, c] = 0
    assert _chi2_over_placements(s, int(t["players"][0]), viewer) == 144


def test_cell_marginals_midgame_standard():
    """every hidden cell of a mid-game Standard state: still cell -> immovable t with n_t / S, movable m with
    (1 - I / S) n_m / M; moved cell -> movable m with n_m / M (chi-square per cell)"""
    states, players = _states("standard")
    vw = np.ones(len(states), dtype=np.int64)
    hidden, still, _, true = hidden_cells(states, players, vw)
    moved = (hidden & ~still).sum(1)
    i = int(np.argmax(np.where(moved >= 3, hidden.sum(1), 0)))
    assert moved[i] >= 3 and hidden[i].sum() >= 20
    n = 100_000
    samples, _ = sample_hidden_ref(states[i:i + 1], players[i:i + 1], vw[i:i + 1], n, seed=77, draw=3)
    cells = np.flatnonzero(hidden[i])
    got = samples.reshape(n, 34, -1)[:, 1][:, cells]
    cnt = code_counts(hidden[i:i + 1], true[i:i + 1])[0].astype(np.float64)
    S, I = still[i].sum(), cnt[FLAG] + cnt[BOMB]
    M = cnt[1:11].sum()
    for j, c in enumerate(cells):
        if still[i, c]:
            prob = np.concatenate([(1 - I / S) * cnt[1:11] / M, cnt[11:13] / S])
        else:
            prob = np.concatenate([cnt[1:11] / M, [0.0, 0.0]])
        obs = np.bincount(got[:, j], minlength=13)[1:13]
        assert obs[prob == 0].sum() == 0
        keep = prob > 0
        p = scipy.stats.chisquare(obs[keep], prob[keep] * n).pvalue
        assert p > P_MIN, (c, bool(still[i, c]), p)


# ---- draw independence ----------------------------------------------------------------------------------------------
def test_sample_k_does_not_depend_on_n_samples_split_or_placement():
    states, players = _states("standard", stride=7)
    B = states.shape[0]
    vw = np.where(np.arange(B) % 3 == 0, 1, -1)
    seed, draw, base = 0xFEDC_BA98_7654_3210, 2 ** 32 - 2, 2 ** 32 - 40
    full, _ = sample_hidden_ref(states, players, vw, 5, seed, draw, env_base=base)
    few, _ = sample_hidden_ref(states, players, vw, 2, seed, draw, env_base=base)
    assert np.array_equal(full.reshape(B, 5, -1)[:, :2], few.reshape(B, 2, -1))
    h = B // 2
    lo, _ = sample_hidden_ref(states[:h], players[:h], vw[:h], 5, seed, draw, env_base=base)
    hi, _ = sample_hidden_ref(states[h:], players[h:], vw[h:], 5, seed, draw, env_base=base + h)
    assert np.array_equal(np.concatenate([lo, hi]), full)
    b = 11
    one, _ = sample_hidden_ref(states[b:b + 1], players[b:b + 1], vw[b:b + 1], 5, seed, draw, env_base=base + b)
    assert np.array_equal(one, full[b * 5:(b + 1) * 5])
    other, _ = sample_hidden_ref(states, players, vw, 5, seed, draw + 1, env_base=base)
    assert not np.array_equal(other, full)


def test_moved_bomb_with_no_still_cell_left_is_reported():
    """I > S: no consistent placement; the rows are copies and the status is 1"""
    t = traj("barrage")
    s = t["states"][0].astype(np.int64).copy()
    s[33] = 0  # every piece of player -1 has 'moved', the bomb and flag included
    good = t["states"][1].astype(np.int64)
    states = np.stack([s, good])
    players = t["players"][:2].astype(np.int64)
    out, status = sample_hidden_ref(states, players, np.asarray([1, 1]), 3, seed=1)
    assert status.tolist() == [1, 0]
    assert np.array_equal(out[:3], np.repeat(s[None], 3, 0))


# ---- argument checks without a device -------------------------------------------------------------------------------
def _config():
    """a Barrage sx_config made without a device (sx_config_create needs none)"""
    from stratego_env_b200 import _lib
    lib = _lib.load()
    cfg = _cfg("barrage")
    desc = _lib.SxConfigDesc()
    desc.rows, desc.cols, desc.max_turns, desc.usable_rows = 10, 10, 1000, 4
    for i, v in enumerate(_amounts(cfg)):
        desc.piece_amounts[i] = int(v)
    from stratego_env_b200.config import captured_lut, obstacle_map, recent_moves_lut, unit_channel_lut
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


@pytest.mark.parametrize("n_samples,num_envs,same,needle", [
    (0, 4, False, b"n_samples"), (-3, 4, False, b"n_samples"), (1 << 24, 4, False, b"n_samples"),
    (1 << 23, 1 << 40, False, b"overflows"), (4, 2 ** 63 - 1, False, b"overflows"),
    (1, 4, True, b"out.board is st.board")])
def test_abi_refusals(n_samples, num_envs, same, needle):
    lib, cfg, keep = _config()
    try:
        st = _fake_state(0x10000)
        out = st if same else _fake_state(0x20000)
        assert lib.sx_sample_hidden_states(cfg, st, num_envs, 0, None, n_samples, 1, 0, out, None, None) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_refuses_null_tensors():
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        st = _fake_state(0x10000)
        assert lib.sx_sample_hidden_states(cfg, st, 4, 0, None, 1, 1, 0, _lib.SxState(), None, None) != 0
        assert b"null out" in lib.sx_last_error()
        assert lib.sx_sample_hidden_states(None, st, 4, 0, None, 1, 1, 0, _fake_state(0x20000), None, None) != 0
        assert b"null config" in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def _no_device_engine(monkeypatch):
    """a StrategoEngine shell whose every library call or device query fails the test"""
    from stratego_env_b200 import engine

    def touched(*a, **k):
        raise AssertionError("the device or the library was reached before the argument check")
    eng = engine.StrategoEngine.__new__(engine.StrategoEngine)
    eng.lib = type("NoLib", (), {"__getattr__": lambda self, name: touched})()
    eng.device = torch.device("cuda", 0)
    monkeypatch.setattr(torch.cuda, "is_available", touched)
    monkeypatch.setattr(torch.cuda, "current_stream", touched)
    state = engine.DeviceState(torch.zeros(4, 112, dtype=torch.uint8), torch.zeros(4, 8, dtype=torch.int16),
                               torch.zeros(4, 16, dtype=torch.int16))
    return eng, state


@pytest.mark.parametrize("n_samples", [0, -1, 1 << 24, 2.0, True, "3", None])
def test_engine_rejects_bad_n_samples_before_touching_a_device(n_samples, monkeypatch):
    eng, state = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="n_samples"):
        eng.sample_hidden_states(state, n_samples=n_samples)


@pytest.mark.parametrize("viewer", [torch.ones(3, dtype=torch.int8), torch.ones(4, 1, dtype=torch.int8),
                                    torch.ones(4, dtype=torch.float32), torch.ones(4, dtype=torch.bool),
                                    np.ones(4, dtype=np.int8), 1])
def test_engine_rejects_bad_viewer_before_touching_a_device(viewer, monkeypatch):
    eng, state = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="viewer"):
        eng.sample_hidden_states(state, n_samples=2, viewer=viewer)
