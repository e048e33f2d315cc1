"""sx_sample_hidden_states on the device: draw for draw against the numpy reference (tests/_hidden_ref.py), viewer
invariance through the engine, independence of the batch split, playability of the samples, the I > S status, and the
invariants at full size."""
import numpy as np
import pytest
import torch

from _golden import VERSIONS, traj
from _hidden_ref import sample_hidden_ref

pytestmark = pytest.mark.gpu

HIGH_SEED = 0x5EED_0000_0000_0002
HIGH_BASE = 2 ** 32 - 5
RANK, OWNER, REVEALED, STILL, OBST = 0x0F, 0x10, 0x20, 0x40, 0x80


def _engine(version, **kw):
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine
    return StrategoEngine(VERSION_CONFIGS[as_version(version)], device="cuda:0", **kw)


def _selfplay(e, B, steps, auto_reset=False, seed=3, env_base=0):
    """B games played by uniform random moves, game b for its own number of plies in [0, steps) (de-phased): a game's
    action is -1 (rejected, the game untouched) once its plies are done"""
    st = e.alloc_state(B)
    e.reset(st, seed=seed, env_base=env_base, shuffle=True)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=seed, env_base=env_base)
    g = torch.Generator(device="cuda").manual_seed(seed)
    target = torch.randint(0, steps, (B,), generator=g, device="cuda")
    for s in range(steps):
        a = torch.where(target > s, actions, torch.full_like(actions, -1))
        e.step_all(st, a, out, env_base=env_base, auto_reset=auto_reset, sample_next=True, seed=seed, shuffle=True)
        actions = torch.where(target > s, out["next_action"], actions)
    return st


def _viewer(kind, B):
    if kind is None:
        return None
    if kind == "mixed":
        return torch.tensor([1, -1, 5, 0] * (B // 4) + [1] * (B % 4), dtype=torch.int8, device="cuda")
    return torch.full((B,), kind, dtype=torch.int8, device="cuda")


def _check_draws(e, st, viewer, K, seed, draw, env_base):
    samples = e.sample_hidden_states(st, n_samples=K, viewer=viewer, seed=seed, draw=draw, env_base=env_base)
    dense, player = e.export_ref_state(st)
    got, got_player = e.export_ref_state(samples)
    vw = None if viewer is None else viewer.cpu().numpy()
    ref, status = sample_hidden_ref(dense.cpu().numpy(), player.cpu().numpy(), vw, K, seed, draw, env_base)
    assert not status.any()
    got = got.cpu().numpy()
    bad = np.nonzero((got != ref).reshape(got.shape[0], -1).any(1))[0]
    assert bad.size == 0, (bad[:8], got.shape)
    assert np.array_equal(got_player.cpu().numpy(), np.repeat(player.cpu().numpy(), K))
    return samples


@pytest.mark.parametrize("version", VERSIONS)
def test_draw_for_draw_on_self_play(version):
    """viewer None / +1 / -1 / mixed, K = 1, 3, 32, env_base near 2^32, a seed with high bits, draw near 2^32, and
    finished games (no auto-reset on the toy boards)"""
    e = _engine(version)
    for viewer, K, B, seed, draw, base in ((None, 1, 512, 1, 0, 0), (1, 3, 256, HIGH_SEED, 2 ** 32 - 1, HIGH_BASE),
                                           (-1, 3, 256, 7, 5, 11), ("mixed", 32, 64, HIGH_SEED, 2 ** 32 - 2, HIGH_BASE - 30)):
        st = _selfplay(e, B, 60, auto_reset=False, seed=len(version) + K, env_base=base)
        _check_draws(e, st, _viewer(viewer, B), K, seed, draw, base)


@pytest.mark.parametrize("version", VERSIONS)
def test_draw_for_draw_on_imported_states(version):
    """every recorded state of the variant (fresh, mid-game and finished games), imported"""
    t = traj(version)
    e = _engine(version)
    dense = torch.as_tensor(t["states"].astype(np.int64), device="cuda")
    st = e.import_ref_state(dense, torch.as_tensor(t["players"], device="cuda"))
    B = st.num_envs
    _check_draws(e, st, None, 2, 9, 3, 0)
    _check_draws(e, st, _viewer("mixed", B), 3, HIGH_SEED, 2 ** 32 - 1, HIGH_BASE)


def test_draw_for_draw_on_curriculum_starts():
    """games (re)started from a curriculum table through step_all's auto-reset"""
    t = traj("barrage")
    e = _engine("barrage")
    e.set_start_states(torch.as_tensor(t["states"][100:300:7].astype(np.int64)), 0)
    B = 512
    st = e.alloc_state(B)
    e.reset(st, seed=4, shuffle=True)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=4)
    for _ in range(30):
        e.step_all(st, actions, out, auto_reset=True, sample_next=True, seed=4, shuffle=True)
        actions = out["next_action"].clone()
    _check_draws(e, st, None, 4, 21, 1, 1000)


def _hidden_mask(board, aux, viewer, N):
    """[B, N] hidden cells of each compact row (viewer tensor of +1 / -1 or None = player to move)"""
    b = board[:, :N].to(torch.int32)
    to_move = ((aux[:, 2].to(torch.int32) >> 4) & 1)
    side = to_move if viewer is None else torch.where(viewer.to(torch.int32) == 1, 0, 1)
    opp = (side ^ 1)[:, None]
    return ((b & RANK) != 0) & (((b & OWNER) != 0).to(torch.int32) == opp) & ((b & (REVEALED | OBST)) == 0)


def _check_invariants(st, samples, viewer, K, N):
    """only CELL_RANK bits of hidden cells differ; aux and capture list are copies; the hidden multiset is kept; no flag
    or bomb on a moved cell"""
    hid = _hidden_mask(st.board, st.aux, viewer, N)
    ob = st.board.repeat_interleave(K, 0)
    sb = samples.board
    assert torch.equal(samples.aux, st.aux.repeat_interleave(K, 0))
    assert torch.equal(samples.captured, st.captured.repeat_interleave(K, 0))
    diff = (ob ^ sb).to(torch.int32)
    assert int((diff & ~RANK).count_nonzero()) == 0
    hid_k = hid.repeat_interleave(K, 0)
    assert int((diff[:, :N] != 0).logical_and(~hid_k).count_nonzero()) == 0
    o_rank, s_rank = (ob[:, :N].to(torch.int32) & RANK), (sb[:, :N].to(torch.int32) & RANK)
    for t in range(1, 13):
        assert torch.equal(((o_rank == t) & hid_k).sum(1), ((s_rank == t) & hid_k).sum(1)), t
    moved = hid_k & ((sb[:, :N].to(torch.int32) & STILL) == 0)
    assert int((moved & (s_rank >= 11)).count_nonzero()) == 0
    return hid


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode", ["extended", "original"])
@pytest.mark.parametrize("version", ["barrage", "standard", "tiny", "standard2"])
def test_viewer_sees_the_same_game(version, mode, dtype):
    """observe(sample, viewer): partial observation and mask equal the original's byte for byte; the compact rows
    differ only in CELL_RANK bits of hidden cells"""
    e = _engine(version, obs_channel_mode=mode, obs_dtype=dtype)
    B, K = 256, 3
    st = _selfplay(e, B, 80, seed=17)
    viewer = _viewer("mixed", B)
    samples = e.sample_hidden_states(st, n_samples=K, viewer=viewer, seed=5, draw=9)
    _check_invariants(st, samples, viewer, K, e.cells)
    v_k = viewer.repeat_interleave(K)
    o = e.observe(st, viewer, partial=True, full=False, mask=True)
    s = e.observe(samples, v_k, partial=True, full=False, mask=True)
    po_o = o["partial_obs"].repeat_interleave(K, 0).view(torch.int16 if dtype != torch.float32 else torch.int32)
    po_s = s["partial_obs"].view(po_o.dtype)
    assert torch.equal(po_o, po_s)
    assert torch.equal(o["valid_mask"].repeat_interleave(K, 0), s["valid_mask"])
    assert torch.equal(o["player"].repeat_interleave(K, 0), s["player"])


def test_batch_split_and_prefix_give_the_same_rows():
    e = _engine("standard")
    B = 300
    st = _selfplay(e, B, 50, seed=8, env_base=1000)
    full = e.sample_hidden_states(st, n_samples=6, seed=HIGH_SEED, draw=4, env_base=1000)
    h = 137
    lo = e.sample_hidden_states(st.select(0, h), n_samples=6, seed=HIGH_SEED, draw=4, env_base=1000)
    hi = e.sample_hidden_states(st.select(h, B), n_samples=6, seed=HIGH_SEED, draw=4, env_base=1000 + h)
    assert torch.equal(torch.cat([lo.board, hi.board]), full.board)
    few = e.sample_hidden_states(st, n_samples=2, seed=HIGH_SEED, draw=4, env_base=1000)
    assert torch.equal(full.board.view(B, 6, -1)[:, :2], few.board.view(B, 2, -1))
    assert torch.equal(full.captured.view(B, 6, -1)[:, :2], few.captured.view(B, 2, -1))


@pytest.mark.parametrize("version", ["barrage", "standard", "octa_barrage", "fives", "tiny"])
def test_samples_play_on_in_lock_step_with_the_oracle(version):
    """a few hundred sampled games step 100 times through step_all and agree with the oracle at every step.  A game
    that is over (or whose mover is stuck) has only the noop entry [0, 0, A - 1] in its mask; playing it is rejected
    (illegal = 1, the game untouched), as maenv.step rejects it in the reference.  Every other sampled action is legal."""
    from oracle.binding import OracleEnvLogic
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    cfg = VERSION_CONFIGS[as_version(version)]
    orc = OracleEnvLogic(cfg["rows"], cfg["columns"], cfg["piece_amounts"])
    e = _engine(version)
    A = e.spatial_channels
    st = _selfplay(e, 100, 40, seed=2)
    samples = e.sample_hidden_states(st, n_samples=3, seed=6)
    B = samples.num_envs
    out = e.alloc_outputs(B, partial=True, full=False, mask=True, sample=True)
    e.observe(samples, out=out)
    actions = e.sample_valid(out["valid_mask"], seed=6)
    played = 0
    for s in range(100):
        mask0 = out["valid_mask"].reshape(B, -1)
        noop_only = ((mask0.sum(1) == 1) & (mask0[:, A - 1] == 1)).cpu().numpy()
        dense0, player0 = e.export_ref_state(samples)
        e.step_all(samples, actions, out, auto_reset=False, sample_next=True, seed=6)
        dense1, _ = e.export_ref_state(samples)
        d0, p0, d1 = dense0.cpu().numpy(), player0.cpu().numpy(), dense1.cpu().numpy()
        acts = actions.cpu().numpy()
        assert np.array_equal(out["illegal"].cpu().numpy() != 0, noop_only), (version, s)
        assert np.array_equal(d1[noop_only], d0[noop_only])
        for b in range(s % 7, B, 7):
            if noop_only[b]:
                continue
            played += 1
            ns, npl = orc.apply_spatial_action(d0[b], int(p0[b]), int(acts[b]))
            assert np.array_equal(ns, d1[b]), (version, s, b)
            mask, po, _ = orc.current_obs(ns, npl, 1)
            assert np.array_equal(mask.reshape(-1), out["valid_mask"][b].cpu().numpy().reshape(-1)), (version, s, b)
            assert np.array_equal(po.view(np.uint32), out["partial_obs"][b].cpu().numpy().view(np.uint32)), (version, s, b)
        actions = out["next_action"].clone()
    assert played > 100


def test_no_placement_status_and_error():
    """an imported state whose bomb and flag have 'moved' (I > S): status 1, the rows unchanged, the engine raises"""
    from stratego_env_b200 import _lib
    t = traj("barrage")
    bad = t["states"][0].astype(np.int64).copy()
    bad[33] = 0
    dense = torch.as_tensor(np.stack([t["states"][5].astype(np.int64), bad]), device="cuda")
    e = _engine("barrage")
    st = e.import_ref_state(dense, torch.tensor([1, 1], dtype=torch.int8, device="cuda"))
    with pytest.raises(ValueError, match=r"\[1\]"):
        e.sample_hidden_states(st, n_samples=3)
    out = e.sample_hidden_states(st, n_samples=3, check=False)
    assert torch.equal(out.board[3:], st.board[1:].repeat(3, 1))
    status = torch.full((2,), 7, dtype=torch.uint8, device="cuda")
    out2 = e.alloc_state(6)
    _lib.check(e.lib.sx_sample_hidden_states(e._cfg, st.as_struct(), 2, 0, None, 3, 0, 0, out2.as_struct(),
                                             status.data_ptr(), torch.cuda.current_stream().cuda_stream))
    assert status.tolist() == [0, 1]


@pytest.mark.parametrize("version,B", [("barrage", 262_144), ("standard", 131_072)])
def test_full_size(version, B):
    """one call at full size, K = 4: invariants on the device, draws against the reference on 4 096 rows"""
    e = _engine(version)
    K = 4
    st = _selfplay(e, B, 60, seed=12)
    samples = e.sample_hidden_states(st, n_samples=K, seed=HIGH_SEED, draw=77, env_base=HIGH_BASE)
    _check_invariants(st, samples, None, K, e.cells)
    g = torch.Generator(device="cuda").manual_seed(1)
    games = torch.randperm(B, generator=g, device="cuda")[:4096 // K].sort().values
    sub = type(st)(st.board[games], st.aux[games], st.captured[games])
    dense, player = e.export_ref_state(sub)
    gids = games.cpu().numpy().astype(np.uint64) + np.uint64(HIGH_BASE)
    ref, _ = sample_hidden_ref(dense.cpu().numpy(), player.cpu().numpy(), None, K, HIGH_SEED, 77, gids=gids)
    rows = (games[:, None] * K + torch.arange(K, device="cuda")).reshape(-1)
    picked = type(st)(samples.board[rows], samples.aux[rows], samples.captured[rows])
    got, _ = e.export_ref_state(picked)
    assert np.array_equal(got.cpu().numpy(), ref)


def test_batched_env_draws_advance_and_viewer_ids():
    from stratego_env_b200.batched_env import BatchedStrategoEnv
    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=64, seed=3, env_base=5)
    env.reset()
    a = env.sample_hidden_states(2)
    b = env.sample_hidden_states(2)
    assert a.num_envs == 128 and not torch.equal(a.board, b.board)
    c = env.engine.sample_hidden_states(env.state, 2, seed=3, draw=1, env_base=5)
    assert torch.equal(a.board, c.board)
    viewer = torch.full((64,), -1, dtype=torch.int8, device="cuda")
    d = env.sample_hidden_states(1, viewer=viewer)
    o = env.observe(viewer, full=False)
    s = env.engine.observe(d, viewer, partial=True, full=False, mask=True)
    assert torch.equal(o["partial_observation"].view(torch.int32), s["partial_obs"].view(torch.int32))
