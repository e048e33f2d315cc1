"""Observation and mask planes in compressible device memory (sx_device_alloc, StrategoEngine(compressible_outputs=)).

Compression happens between L2 and DRAM and must be invisible: an engine whose planes live in one compressible
allocation and an engine with plain ``torch.empty`` planes play the same seeded games in lock step and must agree byte
for byte (uint8 views) on every output and on the state.  333 games: odd and not a multiple of 32, so the
thread-per-game kernel of the toy boards runs with a tail on the warp-level kernel.  The size bound below which the
engine keeps plain memory is lifted so that these small batches take the compressible path too."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

B = 333


def _engine(version, compressible, max_turns=24, **kw):
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine
    cfg = dict(VERSION_CONFIGS[as_version(version)], max_turns=max_turns)
    eng = StrategoEngine(cfg, device="cuda:0", compressible_outputs=None if compressible else False, **kw)
    eng._COMPRESSIBLE_MIN_BYTES = 0
    return eng


def _live():
    from stratego_env_b200 import _lib
    n = C.c_int64()
    assert _lib.load().sx_device_alloc_info(None, None, None, C.byref(n)) == 0
    return n.value


def _granted(t):
    """the flags sx_device_alloc granted the allocation a plane lives in (None: not a library allocation)"""
    from stratego_env_b200 import _lib
    lib, flags = _lib.load(), C.c_uint32()
    base = t.untyped_storage().data_ptr()
    return flags.value if lib.sx_device_alloc_info(base, None, C.byref(flags), None) == 0 else None


def _same(a, b, what):
    assert a.shape == b.shape and a.dtype == b.dtype, what
    eq = a.contiguous().view(torch.uint8) == b.contiguous().view(torch.uint8)
    assert bool(eq.all()), "%s: %d of %d bytes differ" % (what, int((~eq).sum()), eq.numel())


def _lockstep(ref, eng, full, terminal, baseline=False, steps=48, seed=7):
    st_ref = ref.alloc_state(B)
    ref.reset(st_ref, seed=seed, shuffle=True)
    st = st_ref.clone()
    o_ref = ref.alloc_outputs(B, partial=True, full=full, mask=True, sample=True, terminal=terminal)
    o = eng.alloc_outputs(B, partial=True, full=full, mask=True, sample=True, terminal=terminal)
    assert set(o) == set(o_ref)
    planes = [k for k in o if o[k].dim() > 1]
    assert all(_granted(o_ref[k]) is None for k in planes)  # the reference engine's planes are torch's
    assert len({_granted(o[k]) for k in planes}) == 1 and _granted(o[planes[0]]) is not None
    for k in ("terminal_partial_obs", "terminal_full_obs"):
        if k in o:
            assert not bool(o[k].view(torch.uint8).any())  # zero-filled like alloc_outputs' torch.zeros
    ref.observe(st_ref, out=o_ref, partial=True, full=full, mask=True)
    eng.observe(st, out=o, partial=True, full=full, mask=True)
    for k in o:
        _same(o[k], o_ref[k], "observe " + k)
    actions = ref.sample_valid(o_ref["valid_mask"], seed=seed)
    finished = 0
    for s in range(steps):
        kw = dict(auto_reset=True, sample_next=True, shuffle=True, seed=seed, baseline_kernel=baseline)
        ref.step_all(st_ref, actions, o_ref, **kw)
        eng.step_all(st, actions, o, **kw)
        for k in o:
            _same(o[k], o_ref[k], "step %d %s" % (s, k))
        for name in ("board", "aux", "captured"):
            _same(getattr(st, name), getattr(st_ref, name), "step %d state %s" % (s, name))
        finished += int(o_ref["done"].sum())
        actions = o_ref["next_action"].clone()
    assert finished > 0  # auto-reset and the terminal observations were exercised
    return o


CASES = [("barrage", torch.float32, False), ("barrage", torch.bfloat16, False), ("standard", torch.float32, True),
         ("standard", torch.bfloat16, True), ("micro", torch.float32, False), ("micro", torch.bfloat16, True)]


@pytest.mark.parametrize("version,dtype,full", CASES, ids=["%s-%s-%s" % (v, str(d)[6:], "po_fo" if f else "po")
                                                           for v, d, f in CASES])
@pytest.mark.parametrize("terminal", [False, True], ids=["plain", "terminal"])
def test_compressible_planes_match_plain_planes_byte_for_byte(version, dtype, full, terminal):
    from stratego_env_b200 import _lib
    ref, eng = _engine(version, False, obs_dtype=dtype), _engine(version, True, obs_dtype=dtype)
    o = _lockstep(ref, eng, full, terminal)
    assert eng.outputs_compressed == (_granted(o["partial_obs"]) == _lib.SX_ALLOC_COMPRESSIBLE)
    if not eng.outputs_compressed:
        pytest.skip("the device did not grant compressible memory: only the plain library path was compared")


def test_general_kernel_on_a_toy_board_with_compressible_planes():
    """Micro through the warp-level kernel as well (baseline_kernel), terminal observations included"""
    _lockstep(_engine("micro", False), _engine("micro", True), full=True, terminal=True, baseline=True)


def test_forced_fallback_gives_the_same_bytes():
    """the library's plain-memory path (what a device without compression gets) behind the same engine code"""
    eng = _engine("barrage", True)
    eng._alloc_compressible = False
    o = _lockstep(_engine("barrage", False), eng, full=False, terminal=True)
    assert eng.outputs_compressed is False and _granted(o["partial_obs"]) == 0


def test_outputs_compressed_on_b200_at_the_benchmark_size():
    """the headline layout (Barrage, 262 144 games, PO + mask) gets compressible memory with the default setting, one
    allocation for both planes; compressible_outputs=True insists on it"""
    from stratego_env_b200 import _lib
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine
    if "B200" not in torch.cuda.get_device_name(0):
        pytest.skip("not a B200")
    for value in (None, True):
        eng = StrategoEngine(VERSION_CONFIGS[as_version("barrage")], device="cuda:0", compressible_outputs=value)
        o = eng.alloc_outputs(262144, partial=True, mask=True, sample=True)
        assert eng.outputs_compressed is True
        assert _granted(o["partial_obs"]) == _granted(o["valid_mask"]) == _lib.SX_ALLOC_COMPRESSIBLE
        assert o["partial_obs"].untyped_storage().data_ptr() == o["valid_mask"].untyped_storage().data_ptr()
        del o
    small = eng.alloc_outputs(4, partial=True, mask=True)  # below one 2 MB granule: plain torch memory
    assert eng.outputs_compressed is False and _granted(small["partial_obs"]) is None


def test_launch_shape_follows_the_output_memory():
    """10x10 float32 steps into compressible planes run the shape swept for them (12 warps with one observation,
    7 with both); plain planes, 16-bit observations and the thread-per-game boards keep theirs"""
    def warps(version, compressible, dtype=torch.float32, **kw):
        eng = _engine(version, compressible, obs_dtype=dtype)
        eng.alloc_outputs(B, partial=True, full=kw.get("full", False), mask=True)
        return eng.launch_info(partial=True, full=kw.get("full", False), mask=True)
    if not _engine_compressed():
        pytest.skip("the device did not grant compressible memory")
    for version in ("barrage", "standard"):
        assert warps(version, False)["warps_per_block"] == 8
        assert warps(version, True)["warps_per_block"] == 12
        assert warps(version, False, full=True)["warps_per_block"] == 6
        assert warps(version, True, full=True)["warps_per_block"] == 7
        assert warps(version, True, torch.bfloat16) == warps(version, False, torch.bfloat16)
    assert warps("micro", True) == warps("micro", False) and warps("micro", True)["thread_per_game"] == 1


def _engine_compressed():
    eng = _engine("barrage", True)
    eng.alloc_outputs(B)
    return eng.outputs_compressed


def test_tensors_outlive_the_engine_and_each_allocation_is_freed_once():
    import gc
    from stratego_env_b200 import _lib
    lib = _lib.load()
    gc.collect()
    before = _live()
    eng = _engine("barrage", True)
    st = eng.alloc_state(B)
    eng.reset(st, seed=3, shuffle=True)
    o = eng.alloc_outputs(B, partial=True, full=True, mask=True, terminal=True)
    assert _live() == before + 1  # all planes share one allocation
    eng.observe(st, out=o, partial=True, full=True, mask=True)
    want = {k: v.clone() for k, v in o.items()}
    base = o["partial_obs"].untyped_storage().data_ptr()
    del eng
    gc.collect()
    torch.cuda.synchronize()
    po = o["partial_obs"][5:9]  # a view keeps the allocation alive as well
    for k in o:
        _same(o[k], want[k], k)
    del o
    gc.collect()
    assert _live() == before + 1
    _same(po, want["partial_obs"][5:9], "view")
    del po
    gc.collect()
    assert _live() == before
    assert lib.sx_device_free(C.c_void_p(base)) != 0  # freed already: a second free is refused, not performed


def test_device_allocation_directly():
    from stratego_env_b200 import _lib
    from stratego_env_b200.engine import DeviceAllocation
    lib = _lib.load()
    before = _live()
    for compressible in (True, False):
        a = DeviceAllocation("cuda:0", 3 << 20, compressible=compressible)
        nbytes, flags = C.c_uint64(), C.c_uint32()
        assert lib.sx_device_alloc_info(a.ptr, C.byref(nbytes), C.byref(flags), None) == 0
        assert nbytes.value == 3 << 20 and bool(flags.value) == a.compressed
        if not compressible:
            assert not a.compressed
        t = torch.as_tensor(a, device="cuda:0")
        assert t.dtype == torch.uint8 and t.numel() == 3 << 20 and t.data_ptr() == a.ptr
        t.fill_(0x5A)
        assert int(t.sum()) == 0x5A * (3 << 20)
        del a, t
    assert _live() == before


def test_host_buffer_env_host_outputs_equal_its_device_outputs():
    """sx_host_env's observation and mask planes come from sx_device_alloc (compressible when granted and at least
    2 MB); what it copies to the host is what its device buffers hold"""
    from stratego_env_b200 import _lib
    from stratego_env_b200.engine import load_setup_table
    from stratego_env_b200.host_env import HostBufferEnv
    eng = _engine("barrage", True, max_turns=1000)
    n = 1000  # 26.8 MB of observations, 3.7 MB of mask rows: both above the bound
    env = HostBufferEnv(eng, n, setups=load_setup_table("barrage"), seed=9, partial=True, full=True, mask=True,
                        n_chunks=3)
    try:
        host = env.reset()
        dev = _lib.SxOutputs()
        assert eng.lib.sx_host_env_state(env._handle, C.byref(_lib.SxState()), C.byref(dev)) == 0

        class View:
            def __init__(self, ptr, nbytes):
                self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False),
                                                 "strides": None, "version": 3}
        for step in range(6):
            for k in ("partial_obs", "full_obs", "valid_mask"):
                h = host[k]
                nbytes = h.numel() * h.element_size()
                flags = C.c_uint32()
                assert eng.lib.sx_device_alloc_info(getattr(dev, k), None, C.byref(flags), None) == 0
                d = torch.as_tensor(View(getattr(dev, k), nbytes), device="cuda:0")
                _same(d.cpu(), h.contiguous().view(torch.uint8).reshape(-1), "step %d %s" % (step, k))
                if "B200" in torch.cuda.get_device_name(0):
                    assert flags.value == _lib.SX_ALLOC_COMPRESSIBLE, k
            env.actions.copy_(host["next_action"])
            host = env.step()
    finally:
        env.close()
