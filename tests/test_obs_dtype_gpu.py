"""bfloat16 / float16 observations, differential against the float32 path.

An engine built with obs_dtype = bfloat16 or float16 must write, element for element, the round-to-nearest-even
conversion of what the float32 engine writes for the same state (``f32.to(dtype)``), and everything else -- masks,
scalars, sampled actions, the state itself -- byte for byte what the float32 engine writes.  Both engines play the
same seeded games in lock step.  A batch of 333 games is odd and not a multiple of 32, so the thread-per-game kernel
of the toy boards runs with a tail on the warp-level kernel, and every second 10x10 / 5x5 / 12-cell game row of a
16-bit tensor starts off a 16-byte boundary."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DTYPES = [torch.bfloat16, torch.float16]
OBS = ("partial_obs", "full_obs", "terminal_partial_obs", "terminal_full_obs")
B = 333
SENTINEL = 0x7BCD  # int16 pattern of the guard zone (a finite value in both 16-bit formats)


def _versions():
    from stratego_env_b200.config import VERSION_CONFIGS
    return sorted(v.value for v in VERSION_CONFIGS)


def _engines(version, dtype, mode="extended", normalize=True, max_turns=24):
    """a float32 and a 16-bit engine of one variant; max_turns is cut so that games end (and auto-reset, and render
    their terminal observations) within the steps a test plays"""
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine
    cfg = dict(VERSION_CONFIGS[as_version(version)], max_turns=max_turns)
    kw = dict(device="cuda:0", obs_channel_mode=mode, normalize=normalize)
    return StrategoEngine(cfg, **kw), StrategoEngine(cfg, obs_dtype=dtype, **kw)


def _same16(got, f32, what):
    assert got.dtype != torch.float32, what
    want = f32.to(got.dtype)
    eq = got.view(torch.int16) == want.view(torch.int16)
    assert bool(eq.all()), "%s: %d of %d elements differ" % (what, int((~eq).sum()), eq.numel())


def _compare(o32, o16, st32, st16, what):
    for k, v in o32.items():
        if k in OBS:
            _same16(o16[k], v, "%s %s" % (what, k))
        else:
            assert torch.equal(o16[k], v), "%s %s" % (what, k)
    for a, b, name in ((st32.board, st16.board, "board"), (st32.aux, st16.aux, "aux"), (st32.captured, st16.captured, "cap")):
        assert torch.equal(a, b), "%s state %s" % (what, name)


def _lockstep(e32, e16, full, terminal, baseline, steps=64, seed=11):
    st32 = e32.alloc_state(B)
    e32.reset(st32, seed=seed, shuffle=True)
    st16 = st32.clone()
    o32 = e32.alloc_outputs(B, partial=True, full=full, mask=True, sample=True, terminal=terminal)
    o16 = e16.alloc_outputs(B, partial=True, full=full, mask=True, sample=True, terminal=terminal)
    e32.observe(st32, out=o32, partial=True, full=full, mask=True)
    e16.observe(st16, out=o16, partial=True, full=full, mask=True)
    _compare(o32, o16, st32, st16, "observe")
    actions = e32.sample_valid(o32["valid_mask"], seed=seed)
    finished = 0
    for s in range(steps):
        kw = dict(auto_reset=True, sample_next=True, shuffle=True, seed=seed, baseline_kernel=baseline)
        e32.step_all(st32, actions, o32, **kw)
        e16.step_all(st16, actions, o16, **kw)
        _compare(o32, o16, st32, st16, "step %d" % s)
        finished += int(o32["done"].sum())
        actions = o32["next_action"].clone()
    assert finished > 0  # auto-reset (and the terminal observations) were exercised
    return finished


@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "f16"])
@pytest.mark.parametrize("full", [False, True], ids=["po", "po_fo"])
@pytest.mark.parametrize("mode", ["extended", "original"])
@pytest.mark.parametrize("version", _versions())
def test_lockstep_16bit_equals_cast_float32(version, mode, full, dtype):
    e32, e16 = _engines(version, dtype, mode)
    # the specialised kernels (thread-per-game on the toy boards) without terminal buffers, then the general warp-level
    # kernel with the terminal observations of every finished game
    _lockstep(e32, e16, full, terminal=False, baseline=False)
    _lockstep(e32, e16, full, terminal=True, baseline=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "f16"])
@pytest.mark.parametrize("version", ["micro", "fives", "barrage", "standard"])
def test_lockstep_raw_values_engine(version, dtype):
    """normalize=False: the raw channel values (captured counts up to 8, recent-move codes -3..1) in 16 bits"""
    e32, e16 = _engines(version, dtype, normalize=False)
    _lockstep(e32, e16, full=True, terminal=True, baseline=False, steps=40)


@pytest.mark.parametrize("dtype", DTYPES, ids=["bf16", "f16"])
@pytest.mark.parametrize("mode", ["extended", "original"])
@pytest.mark.parametrize("version", ["micro", "tiny", "fives", "medium", "barrage", "standard2"])
def test_observe_with_any_viewer(version, mode, dtype):
    e32, e16 = _engines(version, dtype, mode, max_turns=1000)
    st = e32.alloc_state(B)
    e32.reset(st, seed=5, shuffle=True)
    o = e32.alloc_outputs(B, partial=False, full=False, mask=False, sample=True)
    acts = e32.sample_valid(e32.valid_mask(st), seed=5)
    for _ in range(12):  # a few moves, so that the views differ from the set-up
        e32.step_all(st, acts, o, sample_next=True, shuffle=True, seed=5)
        acts = o["next_action"].clone()
    viewer = torch.where(torch.rand(B, device="cuda:0", generator=torch.Generator("cuda:0").manual_seed(3)) < 0.5, 1, -1)
    viewer = viewer.to(torch.int8)
    a = e32.observe(st, viewer)
    b = e16.observe(st, viewer)
    for k in ("partial_obs", "full_obs"):
        _same16(b[k], a[k], k)
    assert torch.equal(a["valid_mask"], b["valid_mask"]) and torch.equal(a["player"], b["player"])


def _guarded(like, offset):
    """a contiguous tensor shaped like `like` that starts `offset` elements into a larger sentinel-filled buffer"""
    n = like.numel()
    buf = torch.full((n + 16,), SENTINEL, dtype=torch.int16, device=like.device).view(like.dtype)
    return buf, buf[offset:offset + n].view(like.shape).zero_()  # zero like alloc_outputs' terminal buffers


def _untouched(buf, offset, n, what):
    raw = buf.view(torch.int16)
    assert bool((raw[:offset] == SENTINEL).all()) and bool((raw[offset + n:] == SENTINEL).all()), what


@pytest.mark.parametrize("offset", range(8))
@pytest.mark.parametrize("version,mode", [("micro", "extended"), ("fives", "extended"), ("barrage", "extended"),
                                          ("standard", "original"), ("medium", "original")])
def test_outputs_at_any_element_offset_stay_in_bounds(version, mode, offset):
    """every observation output placed at element offset 0..7 of a sentinel-filled buffer: exact values, and not one
    element outside the slice written (before and after each call)"""
    e32, e16 = _engines(version, torch.bfloat16, mode)
    n = 77
    st32 = e32.alloc_state(n)
    e32.reset(st32, seed=9, shuffle=True)
    st16 = st32.clone()
    o32 = e32.alloc_outputs(n, partial=True, full=True, mask=True, sample=True, terminal=True)
    ref = e16.alloc_outputs(n, partial=True, full=True, mask=True, sample=True, terminal=True)
    o16, bufs = dict(ref), {}
    for k in OBS:
        bufs[k], o16[k] = _guarded(ref[k], offset)
        _untouched(bufs[k], offset, ref[k].numel(), "before " + k)
    e32.observe(st32, out=o32)
    e16.observe(st16, out=o16)
    for k in ("partial_obs", "full_obs"):
        _same16(o16[k], o32[k], "observe " + k)
    acts = e32.sample_valid(o32["valid_mask"], seed=9)
    for s in range(40):
        e32.step_all(st32, acts, o32, auto_reset=True, sample_next=True, shuffle=True, seed=9)
        e16.step_all(st16, acts, o16, auto_reset=True, sample_next=True, shuffle=True, seed=9)
        _compare(o32, o16, st32, st16, "step %d" % s)
        acts = o32["next_action"].clone()
    for k in OBS:
        _untouched(bufs[k], offset, ref[k].numel(), "after " + k)


@pytest.mark.parametrize("version,full", [("barrage", False), ("standard", True), ("fives", False), ("octa_barrage", False),
                                          ("medium", True), ("standard2", False), ("micro", False)])
def test_every_tuning_setting_gives_the_same_bytes(version, full):
    outs = {}
    for warps in (0, 4, 8, 12, 16, 24):
        for issue in (0, 1, 2):
            _, e = _engines(version, torch.bfloat16, max_turns=30)
            e.set_tuning(warps, issue)
            st = e.alloc_state(B)
            e.reset(st, seed=4, shuffle=True)
            o = e.alloc_outputs(B, partial=True, full=full, mask=True, sample=True)
            e.observe(st, out=o)
            acts = e.sample_valid(o["valid_mask"], seed=4)
            for _ in range(30):
                e.step_all(st, acts, o, auto_reset=True, sample_next=True, shuffle=True, seed=4, baseline_kernel=True)
                acts = o["next_action"].clone()
            outs[(warps, issue)] = {k: v.clone() for k, v in o.items()}
    first = outs[(0, 0)]
    for key, o in outs.items():
        for k, v in o.items():
            assert torch.equal(v.view(torch.uint8), first[k].view(torch.uint8)), (key, k)


@pytest.mark.parametrize("version,full", [("barrage", False), ("fives", True), ("micro", False)])
def test_host_buffer_env_bf16(version, full):
    """HostBufferEnv of a bf16 engine: pinned bf16 buffers, half the observation bytes per step, and host tensors equal
    to the float32 run cast to bf16 and to the device-resident bf16 observation of the same games"""
    from stratego_env_b200.host_env import HostBufferEnv
    e32, e16 = _engines(version, torch.bfloat16, max_turns=30)
    n = 301
    h32 = HostBufferEnv(e32, n, seed=21, partial=True, full=full, n_chunks=3)
    h16 = HostBufferEnv(e16, n, seed=21, partial=True, full=full, n_chunks=3)
    obs_keys = ["partial_obs"] + (["full_obs"] if full else [])
    assert all(h16.host[k].dtype == torch.bfloat16 and h16.host[k].is_pinned() for k in obs_keys)
    saved = sum(h32.host[k].numel() * 2 for k in obs_keys)
    assert h32.d2h_bytes_per_step - h16.d2h_bytes_per_step == saved
    r32, r16 = h32.reset(), h16.reset()
    for s in range(40):
        for k in r32:
            if k in obs_keys:
                _same16(r16[k], r32[k], "host step %d %s" % (s, k))
            else:
                assert torch.equal(r16[k], r32[k]), (s, k)
        dev = e16.observe(h16.device_state(), partial=True, full=full, mask=True)
        for k in obs_keys:
            assert torch.equal(dev[k].cpu().view(torch.int16), r16[k].view(torch.int16)), (s, k)
        acts = r32["next_action"].clone()
        r32, r16 = h32.step(acts), h16.step(acts)
    h32.close()
    h16.close()


def test_batched_env_bf16_observations():
    """the env-level API: bf16 observation tensors, and the same games as the float32 env"""
    from stratego_env_b200 import BatchedStrategoEnv, GameVersions, ObservationModes
    cfg = {"version": GameVersions.BARRAGE, "observation_mode": ObservationModes.BOTH_OBSERVATIONS}
    a = BatchedStrategoEnv(cfg, num_envs=99, device="cuda:0", seed=2, sample_actions=True)
    b = BatchedStrategoEnv(cfg, num_envs=99, device="cuda:0", seed=2, sample_actions=True, obs_dtype=torch.bfloat16)
    oa, ob = a.reset(), b.reset()
    for _ in range(20):
        for k in ("partial_observation", "full_observation"):
            _same16(ob[k], oa[k], k)
        assert torch.equal(oa["valid_actions_mask"], ob["valid_actions_mask"])
        oa, *_ = a.step(oa["sampled_action"])
        ob, *_ = b.step(ob["sampled_action"])
    wrong = a.engine.alloc_outputs(99, partial=True, full=False, mask=True)
    with pytest.raises(ValueError, match="observations"):
        b.engine.observe(b.state, out=wrong, full=False)
    assert np.array_equal(a.export_states()[0].cpu().numpy(), b.export_states()[0].cpu().numpy())
