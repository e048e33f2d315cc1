"""sx_count_moves / sx_expand_moves on the device: every child, action, count and scalar against the composition it
replaces (valid_mask -> nonzero without the noop channel -> gather -> sx_step), the children against the oracle, the
endings a child can have, determinized worlds, the handling of caller-made offsets, and the full-size batch."""
import numpy as np
import pytest
import torch

from _expand_ref import expand_ref, logic
from _golden import VERSIONS, traj

pytestmark = pytest.mark.gpu

RANK, OWNER = 0x0F, 0x10
FLAG = 11


def _engine(version, **kw):
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine
    return StrategoEngine(VERSION_CONFIGS[as_version(version)], device="cuda:0", **kw)


def _selfplay(e, B, steps, auto_reset=False, seed=3):
    """B games played by uniform random moves, game b for its own number of plies in [0, steps) (de-phased): a game's
    action is -1 (rejected, the game untouched) once its plies are done"""
    st = e.alloc_state(B)
    e.reset(st, seed=seed, shuffle=True)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=seed)
    g = torch.Generator(device="cuda").manual_seed(seed)
    target = torch.randint(0, steps, (B,), generator=g, device="cuda")
    for s in range(steps):
        a = torch.where(target > s, actions, torch.full_like(actions, -1))
        e.step_all(st, a, out, auto_reset=auto_reset, sample_next=True, seed=seed, shuffle=True)
        actions = torch.where(target > s, out["next_action"], actions)
    return st


def _composition(e, st):
    """the five-step composition: mask, nonzero without the noop channel, gather, sx_step on the gathered rows"""
    from stratego_env_b200.engine import DeviceState
    B, A = st.num_envs, e.spatial_channels
    mask = e.valid_mask(st)
    mask[..., A - 1] = 0
    b, idx = torch.nonzero(mask.reshape(B, -1), as_tuple=True)
    kids = DeviceState(st.board.index_select(0, b), st.aux.index_select(0, b), st.captured.index_select(0, b))
    actions = idx.to(torch.int32)
    out = e.step(kids, actions)
    counts = torch.bincount(b, minlength=B)
    return kids, actions, b, counts, out


SCALARS = ("reward", "done", "winner", "ending_invalid", "illegal", "player")


def _check_against_composition(e, st):
    ex = e.expand_moves(st)
    kids, actions, parent, counts, out = _composition(e, st)
    assert torch.equal(ex.offsets[1:] - ex.offsets[:-1], counts)
    assert ex.offsets[0].item() == 0
    assert torch.equal(ex.actions, actions)
    assert torch.equal(ex.parent, parent)
    for name in ("board", "aux", "captured"):
        got, want = getattr(ex.states, name), getattr(kids, name)
        bad = torch.nonzero((got != want).reshape(got.shape[0], -1).any(1)).flatten()
        assert bad.numel() == 0, (name, bad[:8].tolist())
    for name in SCALARS:
        assert torch.equal(getattr(ex, name), out[name]), name
    return ex


def _import(e, t, flip=False):
    dense = torch.as_tensor(t["states"].astype(np.int64), device="cuda")
    player = torch.as_tensor(t["players"].astype(np.int8), device="cuda")
    return e.import_ref_state(dense, -player if flip else player)


@pytest.mark.parametrize("version", VERSIONS)
def test_recorded_states_equal_the_composition(version):
    """every recorded state of the variant (fresh, mid-game, finished), with the recorded and the other player to move"""
    e = _engine(version)
    t = traj(version)
    for flip in (False, True):
        _check_against_composition(e, _import(e, t, flip))


@pytest.mark.parametrize("version", VERSIONS)
def test_self_play_states_equal_the_composition(version):
    """de-phased self-play with and without auto-reset; without it the toy boards hold finished games"""
    e = _engine(version)
    for auto_reset in (False, True):
        st = _selfplay(e, 2048, 150, auto_reset=auto_reset, seed=5 + auto_reset)
        ex = _check_against_composition(e, st)
        assert ex.states.num_envs > 0


@pytest.mark.parametrize("version", ["barrage", "standard", "short_standard"])
@pytest.mark.parametrize("compact", [0, 1])
def test_compact_movers_on_and_off(version, compact):
    """the 10x10 instantiations with the mover hand-out of gen_moves on and off"""
    e = _engine(version)
    e.set_tuning(compact_movers=compact)
    _check_against_composition(e, _selfplay(e, 4096, 200, seed=11))


@pytest.mark.parametrize("version", VERSIONS)
def test_children_equal_the_oracle(version):
    """export_ref_state of the children equals the oracle's step of each listed move, on the recorded states with both
    players to move"""
    e = _engine(version)
    t = traj(version)
    orc = logic(version)
    states = t["states"].astype(np.int64)
    for flip in (False, True):
        players = -t["players"].astype(np.int64) if flip else t["players"].astype(np.int64)
        ex = e.expand_moves(_import(e, t, flip))
        dense, nxt = (x.cpu().numpy() for x in e.export_ref_state(ex.states))
        offsets, actions = ex.offsets.cpu().numpy(), ex.actions.cpu().numpy()
        for i in range(states.shape[0]):
            acts, kids, kid_players = expand_ref(orc, states[i], players[i])
            lo, hi = offsets[i], offsets[i + 1]
            assert np.array_equal(actions[lo:hi], acts), (version, flip, i)
            assert np.array_equal(dense[lo:hi], kids), (version, flip, i)
            assert np.array_equal(nxt[lo:hi], kid_players), (version, flip, i)


def _side(player):
    return torch.where(player == 1, 0, 1)


def test_flag_capture_and_stuck_opponent_children_occur():
    """Micro self-play: children that take the flag and children that leave the opponent without a move both occur
    (the mover wins, reward for player +1 = the winner), and equal the composition"""
    e = _engine("micro")
    st = _selfplay(e, 4096, 12, seed=21)
    ex = _check_against_composition(e, st)
    mover = -ex.player.long()  # the player who made the move
    opp_side = _side(-mover).to(torch.uint8)
    board = ex.states.board[:, :e.cells]
    flag_left = ((board & RANK) == FLAG) & (((board & OWNER) >> 4) == opp_side[:, None])
    won = (ex.done == 1) & (ex.winner.long() == mover) & (ex.ending_invalid == 0)
    took_flag = won & ~flag_left.any(1)
    stuck = won & flag_left.any(1)
    assert int(took_flag.sum()) > 0 and int(stuck.sum()) > 0
    assert torch.equal(ex.reward[won], ex.winner[won].float())


@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_turn_limit_children(version):
    """parents one ply before max_turns: every child that neither takes the flag nor leaves the opponent stuck ends as
    an invalid game with reward 0"""
    e = _engine(version)
    st = _selfplay(e, 1024, 8, seed=4)
    max_turns = int(e.game_version_config["max_turns"])
    st.aux[:, 0] = max_turns - 1
    ex = _check_against_composition(e, st)
    assert ex.states.num_envs > 0
    assert bool((ex.done == 1).all())
    inv = ex.ending_invalid == 1
    assert int(inv.sum()) > 0
    assert bool((ex.reward[inv] == 0).all()) and bool((ex.winner[inv] == 0).all())


def test_finished_parents_have_no_children():
    e = _engine("micro")
    st = _selfplay(e, 2048, 30, seed=8)
    over = (st.aux[:, 2] & 1) == 1  # aux word 1, low byte: the flags, bit 0 = game over
    ex = e.expand_moves(st)
    counts = ex.offsets[1:] - ex.offsets[:-1]
    assert int(over.sum()) > 0
    assert bool((counts[over] == 0).all())


def test_capture_list_overflow_children():
    """a capture list of 8 entries (capture_capacity 1 rounds up to 8): children whose capture does not fit, or whose
    parent's list has overflowed, report illegal = 2, like sx_step"""
    e = _engine("standard", capture_capacity=1)
    ex = _check_against_composition(e, _selfplay(e, 4096, 300, seed=9))
    assert int((ex.illegal == 2).sum()) > 0
    assert bool(((ex.illegal == 0) | (ex.illegal == 2)).all())


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_determinized_worlds_share_the_action_list(version):
    """the K worlds of a game (viewer = player to move) have the parent's action list"""
    e = _engine(version)
    B, K = 512, 8
    st = _selfplay(e, B, 120, seed=13)
    ex = e.expand_moves(st)
    worlds = e.sample_hidden_states(st, n_samples=K, seed=3)
    ew = e.expand_moves(worlds)
    counts = ex.offsets[1:] - ex.offsets[:-1]
    assert torch.equal((ew.offsets[1:] - ew.offsets[:-1]).view(B, K), counts[:, None].expand(B, K))
    game = ew.parent // K
    j = torch.arange(ew.actions.numel(), device="cuda") - ew.offsets[ew.parent]
    assert torch.equal(ew.actions, ex.actions[ex.offsets[game] + j])


def test_caller_offsets_are_respected():
    """a short slot, a long slot, a slot that starts below 0, an empty slot and n_children below the total: exactly the
    rows start + t (t below the count and the slot, inside [0, n_children)) are written, every other row keeps its
    sentinel"""
    from stratego_env_b200 import _lib
    e = _engine("barrage")
    B = 64
    st = _selfplay(e, B, 40, seed=17)
    ref = e.expand_moves(st)
    counts = (ref.offsets[1:] - ref.offsets[:-1]).cpu().numpy()
    assert (counts >= 4).sum() >= 4
    slots = counts.copy()
    big = np.flatnonzero(counts >= 4)
    slots[big[0]] = counts[big[0]] - 3   # short
    slots[big[1]] = counts[big[1]] + 5   # long: rows beyond the count stay untouched
    slots[big[2]] = 0                    # empty
    offsets = np.zeros(B + 1, np.int64)
    offsets[1:] = np.cumsum(slots)
    offsets -= 2                         # game 0's slot starts at -2
    n_children = int(offsets[-1]) - 7    # the last rows are out of range
    cap_rows = int(offsets[-1]) + 16
    out = e.alloc_state(cap_rows)
    for t in (out.board, out.aux, out.captured):
        t.fill_(0x5A)
    sentinel = out.clone()
    actions = torch.full((cap_rows,), -7, dtype=torch.int32, device="cuda")
    scalars = e.alloc_outputs(cap_rows, partial=False, full=False, mask=False)
    for t in scalars.values():
        t.fill_(3)
    off_d = torch.as_tensor(offsets, device="cuda")
    _lib.check(e.lib.sx_expand_moves(e._cfg, st.as_struct(), B, off_d.data_ptr(), n_children, out.as_struct(),
                                     actions.data_ptr(), e._outputs_struct(scalars), torch.cuda.current_stream().cuda_stream),
               "sx_expand_moves")
    written = np.zeros(cap_rows, bool)
    src = np.full(cap_rows, -1, np.int64)  # row of `ref` each written row must equal
    ref_off = ref.offsets.cpu().numpy()
    for b in range(B):
        for t in range(min(counts[b], slots[b])):
            row = offsets[b] + t
            if 0 <= row < n_children:
                written[row], src[row] = True, ref_off[b] + t
    assert written.sum() > 0 and (~written).sum() > 16
    w, s = torch.as_tensor(np.flatnonzero(written), device="cuda"), torch.as_tensor(src[written], device="cuda")
    u = torch.as_tensor(np.flatnonzero(~written), device="cuda")
    assert torch.equal(actions[w], ref.actions[s]) and bool((actions[u] == -7).all())
    for name in ("board", "aux", "captured"):
        got, want = getattr(out, name), getattr(ref.states, name)
        assert torch.equal(got[w], want[s]), name
        assert torch.equal(got[u], getattr(sentinel, name)[u]), name
    for name in SCALARS:
        assert torch.equal(scalars[name][w], getattr(ref, name)[s]), name
        assert bool((scalars[name][u] == 3).all()), name


def test_full_size_barrage_equals_the_composition():
    """262 144 de-phased Barrage games: millions of children, byte for byte"""
    e = _engine("barrage")
    ex = _check_against_composition(e, _selfplay(e, 262144, 120, seed=1))
    assert ex.states.num_envs > 1_000_000
