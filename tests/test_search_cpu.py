"""No-GPU checks of the device tree search (sx_search): the reference of tests/_search_ref.py on recorded states of
several variants (the contract's consequences), max_nodes = 1 as independent playouts, the argument checks of the C ABI
and of StrategoEngine.search before any device is touched."""
import math

import numpy as np
import pytest

from _expand_ref import action_list, logic
from _golden import traj
from _playout_ref import OVER, data
from _search_ref import FIELDS, check_invariants, outcome, score, search_playout, search_ref
from test_expand_moves_cpu import _config, _fake_state, _no_device_engine, _state

SEED = 0x1234_5678_9ABC_DEF0  # non-zero high word
GID0 = 3 << 32                 # gids above 2^32


def _picks(t, k):
    """k recorded states spread over the trajectory, the first of them a game start"""
    n = t["states"].shape[0]
    return sorted({int(np.flatnonzero(t["game_start"])[0]), *np.linspace(0, n - 1, k).astype(int).tolist()})


@pytest.mark.parametrize("version", ["barrage", "standard", "fives", "micro"])
def test_reference_invariants(version):
    """root N = iterations, N = 1 + the children's N on expanded non-root nodes and their sum on the root, children in
    ascending action order and equal to the expand action list, a result that depends on nothing but its inputs"""
    t = traj(version)
    orc = logic(version)
    for i in _picks(t, 4):
        st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
        tree = search_ref(orc, st, pl, GID0 + i, SEED, 48, 1 + 32 * 48, 24, 1.0)
        check_invariants(tree, 48, 1 + 32 * 48)
        if tree["first_child"][0] >= 0:
            f, n = tree["first_child"][0], tree["n_children"][0]
            assert np.array_equal(tree["action"][f:f + n], action_list(orc, st, pl)), (version, i)
        else:
            assert data(st, OVER) or len(action_list(orc, st, pl)) == 0, (version, i)
        again = search_ref(orc, st, pl, GID0 + i, SEED, 48, 1 + 32 * 48, 24, 1.0)
        assert all(np.array_equal(tree[k], again[k]) for k in FIELDS), (version, i)


@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_small_pools_and_zero_iterations(version):
    """a pool too small for a second expansion stops growing, and iterations = 0 leaves the root alone"""
    t = traj(version)
    orc = logic(version)
    i = _picks(t, 2)[0]
    st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
    n = len(action_list(orc, st, pl))
    tree = search_ref(orc, st, pl, GID0, SEED, 40, 1 + n, 8, 1.0)
    check_invariants(tree, 40, 1 + n)
    assert tree["used"] == 1 + n and np.all(tree["first_child"][1:] == -1)
    empty = search_ref(orc, st, pl, GID0, SEED, 0, 10, 8, 1.0)
    assert empty["used"] == 1 and empty["visits"][0] == 0 and empty["value"][0] == 0


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_one_node_is_independent_playouts(version):
    """max_nodes = 1: the root is never expanded, and its W is the sum of `iterations` playouts of the root, playout i
    drawn with RNG_SEARCH ^ i"""
    t = traj(version)
    orc = logic(version)
    for i in _picks(t, 3):
        st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
        tree = search_ref(orc, st, pl, GID0 + i, SEED, 12, 1, 40, 1.0)
        assert tree["used"] == 1 and tree["visits"][0] == 12 and tree["first_child"][0] == -1
        if data(st, OVER):
            want = 12 * outcome(st)
        else:
            want = sum(search_playout(orc, st, pl, GID0 + i, it, SEED, 40)[0] for it in range(12))
        assert tree["value"][0] == want, (version, i)


def test_scores_are_float32_and_break_ties_low():
    """the score is computed in float32 with one rounding per operation; equal scores go to the lowest index"""
    s = score([1, 1, -2], [3, 3, 5], 11, 1, 1.4)
    f = np.float32
    q0 = f(1) / f(3)
    u0 = (f(1.4) * np.sqrt(f(11))) / f(4)
    assert s.dtype == np.float32 and s[0] == f(q0 + u0) and s[0] == s[1] and int(np.argmax(s)) == 0
    assert score([2], [4], 9, -1, 0.0)[0] == f(-0.5)


# ---- argument checks without a device -------------------------------------------------------------------------------
def _tree(**null):
    from stratego_env_b200 import _lib
    names = [n for n, _ in _lib.SxTree._fields_]
    return _lib.SxTree(*(None if null.get(n) else 0x70000 + 0x1000 * k for k, n in enumerate(names)))


def _search_call(lib, cfg, st=None, num_envs=4, iterations=8, max_nodes=64, max_plies=5, c_explore=1.0, tree=None):
    return lib.sx_search(cfg, _fake_state(0x10000) if st is None else st, num_envs, 0, iterations, max_nodes, max_plies,
                         c_explore, 1, _tree() if tree is None else tree, None)


@pytest.mark.parametrize("case,kw,needle", [
    ("null config", {}, b"null config"),
    ("null state", {"st": "null"}, b"null state"),
    *[("null " + n, {"tree": n}, b"null tree") for n in ("visits", "value", "parent", "first_child", "n_children",
                                                          "action", "used")],
    ("negative iterations", {"iterations": -1}, b"iterations"),
    ("iterations above 2^24", {"iterations": (1 << 24) + 1}, b"iterations"),
    ("zero max_nodes", {"max_nodes": 0}, b"max_nodes"),
    ("negative max_nodes", {"max_nodes": -5}, b"max_nodes"),
    ("negative max_plies", {"max_plies": -1}, b"max_plies"),
    ("negative c_explore", {"c_explore": -0.5}, b"c_explore"),
    ("nan c_explore", {"c_explore": math.nan}, b"c_explore"),
    ("inf c_explore", {"c_explore": math.inf}, b"c_explore"),
])
def test_abi_refusals(case, kw, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        kw = dict(kw)
        if kw.get("st") == "null":
            kw["st"] = _lib.SxState()
        if "tree" in kw:
            kw["tree"] = _tree(**{kw["tree"]: True})
        assert _search_call(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_no_games_is_a_no_op():
    """num_envs <= 0 launches nothing (the fake pointers are never touched); the limits of every argument pass"""
    lib, cfg, keep = _config()
    try:
        for n in (0, -3):
            for it, nodes, plies, c in ((0, 1, 0, 0.0), (1 << 24, (1 << 31) - 1, (1 << 31) - 1, 3.0e38)):
                assert _search_call(lib, cfg, num_envs=n, iterations=it, max_nodes=nodes, max_plies=plies,
                                    c_explore=c) == 0, lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


@pytest.mark.parametrize("state", [None, "state", (1, 2, 3), _state()], ids=["None", "str", "tuple", "host tensors"])
def test_engine_rejects_bad_state_before_touching_a_device(state, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="state"):
        eng.search(state, 8)


BAD_INTS = [-1, True, False, 1.0, 2.5, "7", None]


@pytest.mark.parametrize("iterations", BAD_INTS + [(1 << 24) + 1, 1 << 40])
def test_engine_rejects_bad_iterations_before_touching_a_device(iterations, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="iterations"):
        eng.search(_state(), iterations)


@pytest.mark.parametrize("max_nodes", [0, -1, True, 1.0, "7", 1 << 31])
def test_engine_rejects_bad_max_nodes_before_touching_a_device(max_nodes, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="max_nodes"):
        eng.search(_state(), 8, max_nodes=max_nodes)


@pytest.mark.parametrize("max_plies", [-1, True, False, 1.0, 2.5, "7", 1 << 31, 1 << 40])
def test_engine_rejects_bad_max_plies_before_touching_a_device(max_plies, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="max_plies"):
        eng.search(_state(), 8, max_plies=max_plies)


@pytest.mark.parametrize("c_explore", [-0.1, math.nan, math.inf, -math.inf, 1e39, True, "1", None])
def test_engine_rejects_bad_c_explore_before_touching_a_device(c_explore, monkeypatch):
    eng = _no_device_engine(monkeypatch)
    with pytest.raises(ValueError, match="c_explore"):
        eng.search(_state(), 8, c_explore=c_explore)

