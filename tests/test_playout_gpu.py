"""sx_playout on the device, byte for byte against the chain of fused steps it stands for (board with padding, aux,
capture list, the six scalars and the plies), on recorded, self-play, determinized and expanded states of every
variant; ply caps and composition, continuing a step_all chain, gid and seed handling, the CPU reference, and the
full-size batches."""
import numpy as np
import pytest
import torch

from _expand_ref import logic
from _golden import VERSIONS, traj
from _playout_ref import playout_ref
from _sampler_ref import step_words, uniform_valid_ref
from test_expand_moves_gpu import _engine, _import, _selfplay

pytestmark = pytest.mark.gpu

SCALARS = ("reward", "done", "winner", "ending_invalid", "illegal", "player")
STATE = ("board", "aux", "captured")


def _flags(st):
    return st.aux[:, 2].long() & 0xFF  # aux word 1, low byte (aux_pack, sx_device.cuh)


def _first_action(e, st, seed, env_base):
    """the SX_SAMPLE_NEXT draw on each game's current state (_sampler_ref over the valid mask of the player to move)"""
    B = st.num_envs
    mask = e.valid_mask(st).reshape(B, -1).cpu().numpy()
    aux = st.aux.cpu().numpy().view(np.uint16).astype(np.uint64)
    episode = aux[:, 6] | (aux[:, 7] << np.uint64(16))
    words = step_words(np.uint64(env_base) + np.arange(B, dtype=np.uint64), aux[:, 0], episode, seed)
    return torch.as_tensor(uniform_valid_ref(mask, words), dtype=torch.int32, device="cuda")


def _chain(e, st, n, seed, env_base=0):
    """what a playout of at most n plies (None: to the end) stands for: step_all(a, sample_next, no auto-reset) with
    a = next_action, from the draw on the initial state; each game's rows and scalars are kept from the step where done
    first appears.  A player to move without a move at entry instead plays one step of the 1D noop (and loses).
    Returns (final state, scalars, plies, over at entry); the state rows of games over at entry are not meaningful, and
    the scalars of a game no step was kept for are its entry scalars."""
    from stratego_env_b200.engine import DeviceState
    B, A = st.num_envs, e.spatial_channels
    cur = st.clone()
    over0 = (_flags(st) & 1) == 1
    mask = e.valid_mask(cur).reshape(B, -1)
    stuck = ~over0 & (mask.sum(1) == 1) & (mask[:, A - 1] == 1)
    a = _first_action(e, cur, seed, env_base)
    final = cur.clone()
    scalars = _aux_scalars(st)
    plies = torch.zeros(B, dtype=torch.int32, device="cuda")
    fin = over0.clone()

    def keep(rows, state, out):
        for name in STATE:
            setattr(final, name, torch.where(rows[:, None], getattr(state, name), getattr(final, name)))
        for name in SCALARS:
            scalars[name] = torch.where(rows, out[name], scalars[name])

    if bool(stuck.any()):
        tmp = cur.clone()
        out = e.step(tmp, torch.full((B,), e.action_size - 1, dtype=torch.int32, device="cuda"), one_d=True)
        keep(stuck, tmp, out)
        plies += stuck.to(torch.int32)
        fin |= stuck
    out = e.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    steps = 0
    while n is None or steps < n:
        if n is None and steps % 64 == 0 and bool(fin.all()):
            break
        e.step_all(cur, a, out, sample_next=True, seed=seed, env_base=env_base)
        live = ~fin
        keep(live, cur, out)
        plies += live.to(torch.int32)
        fin = fin | (out["done"] == 1)
        a = out["next_action"].clone()
        steps += 1
    return DeviceState(final.board, final.aux, final.captured), scalars, plies, over0


def _aux_scalars(st):
    """the scalars a playout reports for a game it plays no ply of (over at entry, or max_plies = 0), from its aux"""
    f = _flags(st)
    done = f & 1
    winner = torch.where(done == 1, ((f >> 2) & 3) - 1, 0)
    invalid = done * ((f >> 1) & 1)
    return {"done": done.to(torch.uint8), "winner": winner.to(torch.int8), "ending_invalid": invalid.to(torch.uint8),
            "illegal": (2 * ((f >> 5) & 1)).to(torch.uint8), "reward": torch.where(invalid == 1, 0, winner).float(),
            "player": torch.where(((f >> 4) & 1) == 0, 1, -1).to(torch.int8)}


def _check(e, st, n, seed=7, env_base=0):
    """playout of a copy of st against the chain, byte for byte; games over at entry against their input"""
    want, want_sc, want_plies, over0 = _chain(e, st, n, seed, env_base)
    got = st.clone()
    res = e.playout(got, max_plies=n, seed=seed, env_base=env_base)
    live = ~over0
    for name in STATE:
        g, w, s = getattr(got, name), getattr(want, name), getattr(st, name)
        bad = torch.nonzero((g[live] != w[live]).reshape(int(live.sum()), -1).any(1)).flatten()
        assert bad.numel() == 0, (name, bad[:8].tolist())
        assert torch.equal(g[over0], s[over0]), name
    assert torch.equal(res.plies[live], want_plies[live])
    assert bool((res.plies[over0] == 0).all())
    for name in SCALARS:
        assert torch.equal(getattr(res, name), want_sc[name]), name
    return got, res


@pytest.mark.parametrize("version", VERSIONS)
def test_recorded_states_equal_the_chain(version):
    """every recorded state (fresh, mid-game, finished), with the recorded and the other player to move, to the end"""
    e = _engine(version)
    t = traj(version)
    for flip in (False, True):
        _check(e, _import(e, t, flip), None)


@pytest.mark.parametrize("version", VERSIONS)
def test_self_play_states_equal_the_chain(version):
    """de-phased self-play with and without auto-reset (without it the batch holds finished games), to the end"""
    e = _engine(version)
    for auto_reset in (False, True):
        st = _selfplay(e, 1024, 150, auto_reset=auto_reset, seed=5 + auto_reset)
        got, res = _check(e, st, None, seed=21)
        assert bool((res.done == 1).all())


@pytest.mark.parametrize("version", VERSIONS)
def test_determinized_worlds_and_children_equal_the_chain(version):
    """the worlds sample_hidden_states draws and the children expand_moves makes, to the end"""
    e = _engine(version)
    st = _selfplay(e, 256, 60, seed=13)
    _check(e, e.sample_hidden_states(st, n_samples=4, seed=3), None, seed=5)
    kids = e.expand_moves(st).states
    _check(e, kids.select(0, min(kids.num_envs, 2048)), None, seed=6)


@pytest.mark.parametrize("version", ["barrage", "standard", "short_standard"])
@pytest.mark.parametrize("compact", [0, 1])
def test_compact_movers_on_and_off(version, compact):
    e = _engine(version)
    e.set_tuning(compact_movers=compact)
    _check(e, _selfplay(e, 2048, 100, seed=11), None, seed=compact)


@pytest.mark.parametrize("version", ["barrage", "standard", "micro", "fives"])
@pytest.mark.parametrize("cap", [0, 1, 7])
def test_ply_caps(version, cap):
    e = _engine(version)
    st = _selfplay(e, 1024, 80, seed=2)
    got, res = _check(e, st, cap)
    assert bool((res.plies <= cap).all())


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_chunked_calls_equal_one_call(version):
    """playout(3), playout(0), playout(1), playout(40), playout(None) equals playout(None)"""
    e = _engine(version)
    st = _selfplay(e, 2048, 50, seed=4)
    whole = st.clone()
    ref = e.playout(whole, seed=9)
    part = st.clone()
    total = torch.zeros_like(ref.plies)
    for cap in (3, 0, 1, 40, None):
        res = e.playout(part, max_plies=cap, seed=9)
        total += res.plies
    for name in STATE:
        assert torch.equal(getattr(part, name), getattr(whole, name)), name
    assert torch.equal(total, ref.plies)
    for name in SCALARS:
        assert torch.equal(getattr(res, name), getattr(ref, name)), name


@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_playout_continues_a_step_all_chain(version):
    """after step_all(sample_next=True, seed=s), playout(seed=s, max_plies=1) plays that step's next_action"""
    e = _engine(version)
    B, s = 1024, 77
    st = _selfplay(e, B, 40, seed=6)
    out = e.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    e.step_all(st, _first_action(e, st, s, 0), out, sample_next=True, seed=s)
    live = (out["done"] == 0) & ((_flags(st) & 1) == 0)  # (a finished game's noop entry is rejected, not done)
    via_step = st.clone()
    e.step_all(via_step, out["next_action"].clone(), e.alloc_outputs(B, partial=False, full=False, mask=False,
                                                                     sample=True), sample_next=True, seed=s)
    via_playout = st.clone()
    res = e.playout(via_playout, max_plies=1, seed=s)
    assert int(live.sum()) > 0
    assert bool((res.plies[live] == 1).all())
    for name in STATE:
        assert torch.equal(getattr(via_playout, name)[live], getattr(via_step, name)[live]), name


def test_gid_and_seed_handling():
    """env_base >= 2^32, a seed with non-zero high bits, 333 games; two half-batch calls with their env_base equal one
    call"""
    e = _engine("barrage")
    base, seed = (5 << 32) + 123, 0xDEAD_BEEF_0000_0011
    st = _selfplay(e, 333, 30, seed=8)
    got, res = _check(e, st, None, seed=seed, env_base=base)
    halves = st.clone()
    r0 = e.playout(halves.select(0, 160), seed=seed, env_base=base)
    r1 = e.playout(halves.select(160, 333), seed=seed, env_base=base + 160)
    for name in STATE:
        assert torch.equal(getattr(halves, name), getattr(got, name)), name
    assert torch.equal(torch.cat([r0.plies, r1.plies]), res.plies)
    other = st.clone()
    e.playout(other, seed=seed ^ (1 << 40), env_base=base)
    assert not torch.equal(other.board, got.board)  # the high seed word is part of the key


@pytest.mark.parametrize("version", VERSIONS)
def test_kernel_equals_the_cpu_reference(version):
    """64 de-phased games per variant played to the end, against _playout_ref on the exported states"""
    e = _engine(version)
    orc = logic(version)
    B, seed, base = 64, 0xABCD_0000_1234, 1 << 33
    st = _selfplay(e, B, 40, seed=12)
    dense, player = (x.cpu().numpy() for x in e.export_ref_state(st))
    episode = st.aux.cpu().numpy().view(np.uint16).astype(np.int64)
    episode = episode[:, 6] | (episode[:, 7] << 16)
    got = st.clone()
    res = e.playout(got, seed=seed, env_base=base)
    gd, gp = (x.cpu().numpy() for x in e.export_ref_state(got))
    plies = res.plies.cpu().numpy()
    done, winner, inv = (getattr(res, n).cpu().numpy() for n in ("done", "winner", "ending_invalid"))
    for b in range(B):
        want, want_player, n, (over, win, invalid) = playout_ref(orc, dense[b], player[b], base + b, episode[b], seed,
                                                                  (1 << 31) - 1)
        assert np.array_equal(gd[b], want) and gp[b] == want_player and plies[b] == n, (version, b)
        assert done[b] == over == 1 and winner[b] == win and inv[b] == invalid, (version, b)


@pytest.mark.parametrize("version,B", [("barrage", 262144), ("standard", 131072)])
def test_full_size_equals_the_chain(version, B):
    """a full-size de-phased batch played to the end, byte for byte"""
    e = _engine(version)
    got, res = _check(e, _selfplay(e, B, 120, seed=1), None, seed=3)
    assert bool((res.done == 1).all())
