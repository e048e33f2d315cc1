"""sx_state_keys on the device: bit for bit against the reference of tests/_keys_ref.py on the exported states, in both
modes and for both viewers and the player to move, on recorded, full-size self-play and expanded states; the bytes
that are not part of the game (episode counter, padding, capture-list order, overflow flag); a position reached by two
move orders; and the worlds sample_hidden_states draws."""
import numpy as np
import pytest
import torch

from _golden import VERSIONS, traj
from _keys_ref import state_keys_ref
from test_expand_moves_gpu import _engine, _import, _selfplay

pytestmark = pytest.mark.gpu

VIEWERS = ("state", 1, -1, None)  # the state key, then the information-set keys of +1, -1 and the player to move


def _keys(e, st, mode):
    if mode == "state":
        return e.state_keys(st)
    viewer = None if mode is None else torch.full((st.num_envs,), mode, dtype=torch.int8, device="cuda")
    return e.state_keys(st, info_set=True, viewer=viewer)


def _check_reference(e, st, chunk=8192):
    """every game's keys in the four modes against the reference on its export (in chunks: the dense export of a
    full-size batch would not fit the host comfortably)"""
    got = {m: _keys(e, st, m).cpu().numpy().view(np.uint64) for m in VIEWERS}
    for lo in range(0, st.num_envs, chunk):
        part = st.select(lo, min(lo + chunk, st.num_envs))
        dense, player = (x.cpu().numpy() for x in e.export_ref_state(part))
        player = player.astype(np.int64)
        B = dense.shape[0]
        for m in VIEWERS:
            want = state_keys_ref(dense, player, info_set=m != "state",
                                  viewer=None if m in ("state", None) else np.full(B, m))
            bad = np.flatnonzero(got[m][lo:lo + B] != want)
            assert bad.size == 0, (m, (lo + bad[:8]).tolist())
    return got


@pytest.mark.parametrize("version", VERSIONS)
def test_recorded_states_equal_the_reference(version):
    e = _engine(version)
    t = traj(version)
    for flip in (False, True):
        _check_reference(e, _import(e, t, flip))


@pytest.mark.parametrize("version,B", [("barrage", 262144), ("standard", 131072), ("micro", 262144)])
def test_full_size_self_play_equals_the_reference(version, B):
    e = _engine(version)
    _check_reference(e, _selfplay(e, B, 150, auto_reset=True, seed=4))


@pytest.mark.parametrize("version", VERSIONS)
def test_children_equal_the_reference(version):
    e = _engine(version)
    kids = e.expand_moves(_selfplay(e, 256, 60, seed=9)).states
    _check_reference(e, kids.select(0, min(kids.num_envs, 8192)))


@pytest.mark.parametrize("version", ["barrage", "standard", "standard2", "micro"])
def test_bytes_outside_the_game_do_not_count(version):
    """episode counter, board padding, capture entries beyond the count, the order of the capture entries and the
    overflow flag are overwritten in place: no key changes, and neither does the export"""
    e = _engine(version)
    st = _selfplay(e, 4096, 200, auto_reset=True, seed=2)
    before = {m: _keys(e, st, m) for m in VIEWERS}
    dense0, player0 = e.export_ref_state(st)
    g = torch.Generator(device="cuda").manual_seed(1)
    B, N = st.num_envs, e.cells
    st.aux[:, 6:8] = torch.randint(-32768, 32767, (B, 2), generator=g, device="cuda", dtype=torch.int16)
    st.aux[:, 2] |= 1 << 5  # the sticky overflow flag
    if st.board.shape[1] > N:
        st.board[:, N:] = torch.randint(0, 256, (B, st.board.shape[1] - N), generator=g, device="cuda",
                                        dtype=torch.int32).to(torch.uint8)
    ncap = (st.aux[:, 2].long() >> 8) & 0xFF
    cap = st.captured.cpu().numpy()
    rng = np.random.default_rng(3)
    permuted = 0
    for b, n in enumerate(ncap.cpu().numpy()):
        cap[b, n:] = rng.integers(-32768, 32767, cap.shape[1] - n)
        if n > 1:
            cap[b, :n] = cap[b, rng.permutation(n)]
            permuted += 1
    assert permuted > 100
    st.captured.copy_(torch.as_tensor(cap))
    dense1, player1 = e.export_ref_state(st)
    assert torch.equal(dense0, dense1) and torch.equal(player0, player1)
    for m in VIEWERS:
        assert torch.equal(_keys(e, st, m), before[m]), m


def test_two_move_orders_reach_one_key():
    """from a fresh Barrage game, the five plies A X C Z B and C X A Z B (A, C, B moves of player +1 and X, Z of player
    -1 from the start position): wherever both orders are legal and reach the same export, they reach the same key, and
    wherever the exports differ, so do the keys; many such transpositions exist"""
    from stratego_env_b200.engine import DeviceState
    e = _engine("barrage")
    s0 = e.alloc_state(1)
    e.reset(s0, seed=5, shuffle=True)
    plus = np.flatnonzero(e.valid_mask(s0).reshape(-1).cpu().numpy())
    plus = plus[plus % e.spatial_channels != e.spatial_channels - 1]
    minus = e.valid_mask(s0, player=torch.tensor([-1], dtype=torch.int8, device="cuda")).reshape(-1).cpu().numpy()
    minus = np.flatnonzero(minus)
    minus = minus[minus % e.spatial_channels != e.spatial_channels - 1]
    rng = np.random.default_rng(0)
    T = 32768
    a, c, bb = (rng.choice(plus, T) for _ in range(3))
    x, z = (rng.choice(minus, T) for _ in range(2))
    keys, exports, legal = [], [], []
    for order in ((a, x, c, z, bb), (c, x, a, z, bb)):
        st = DeviceState(*(t.expand(T, -1).contiguous() for t in (s0.board, s0.aux, s0.captured)))
        ok = torch.ones(T, dtype=torch.bool, device="cuda")
        for act in order:
            out = e.step(st, torch.as_tensor(act, dtype=torch.int32, device="cuda"))
            ok &= (out["illegal"] == 0) & (out["done"] == 0)
        keys.append(e.state_keys(st))
        dense, player = e.export_ref_state(st)
        exports.append(torch.cat([dense.reshape(T, -1), player.long()[:, None]], 1))
        legal.append(ok)
    both = legal[0] & legal[1]
    same_export = (exports[0] == exports[1]).all(1) & both
    same_key = (keys[0] == keys[1]) & both
    assert torch.equal(same_key, same_export)
    assert int((same_export & torch.as_tensor(a != c, device="cuda")).sum()) > 100


@pytest.mark.parametrize("version", VERSIONS)
@pytest.mark.parametrize("viewer", [1, -1, None], ids=["plus", "minus", "mover"])
def test_determinized_worlds_share_the_information_set_key(version, viewer):
    """the K = 64 worlds sample_hidden_states draws for a viewer all have their source's information-set key for that
    viewer; their state keys differ exactly where their boards differ from the source's"""
    e = _engine(version)
    st = _selfplay(e, 512, 80, seed=7)
    B, K = st.num_envs, 64
    view = None if viewer is None else torch.full((B,), viewer, dtype=torch.int8, device="cuda")
    worlds = e.sample_hidden_states(st, n_samples=K, viewer=view, seed=11, check=False)
    wview = None if view is None else view.repeat_interleave(K)
    src = e.state_keys(st, info_set=True, viewer=view).repeat_interleave(K)
    assert torch.equal(e.state_keys(worlds, info_set=True, viewer=wview), src)
    same = (worlds.board == st.board.repeat_interleave(K, 0)).all(1)
    moved = e.state_keys(worlds) != e.state_keys(st).repeat_interleave(K)
    assert torch.equal(moved, ~same)
    if version not in ("micro", "tiny"):
        assert bool(moved.any())


def test_env_keys_are_the_engine_keys():
    from stratego_env_b200.batched_env import BatchedStrategoEnv
    from stratego_env_b200.enums import GameVersions
    env = BatchedStrategoEnv({"version": GameVersions.BARRAGE}, num_envs=64, device="cuda:0", seed=3)
    env.reset()
    assert torch.equal(env.state_keys(), env.engine.state_keys(env.state))
    v = torch.where(torch.arange(64, device="cuda") % 2 == 0, 1, -1).to(torch.int8)
    assert torch.equal(env.state_keys(info_set=True, viewer=v), env.engine.state_keys(env.state, info_set=True, viewer=v))
