"""No-GPU checks of the guided tree search (sx_guided_select / sx_guided_backup): the reference of tests/_guided_ref.py
on recorded states of several variants (the contract's consequences), the float32 score and its tie rule, the argument
checks of the C ABI and of StrategoEngine.guided_tree / guided_select / guided_backup before any device is touched."""
import math

import numpy as np
import pytest
import torch

from _expand_ref import action_list, logic
from _golden import traj
from _guided_ref import (LEAF_EVAL, LEAF_OVER, LOGIT_CASES, GuidedTree, check_invariants, check_priors, net,
                         network_logits, prior_bound, scores, softmax64, softmax_f32)
from _playout_ref import OVER, data
from test_expand_moves_cpu import _config, _fake_state, _no_device_engine, _state


def _picks(t, k):
    """k recorded states spread over the trajectory, the first of them a game start"""
    n = t["states"].shape[0]
    return sorted({int(np.flatnonzero(t["game_start"])[0]), *np.linspace(0, n - 1, k).astype(int).tolist()})


def _grow(orc, st, pl, rounds, max_nodes, c_puct=1.25, fpu=0.0):
    """a reference tree after `rounds` rounds with the test network, and the (node, kind) of every round's leaf"""
    tree = GuidedTree(orc, st, pl, max_nodes)
    n_logits = orc.current_obs(st, pl, obs_mode=0)[0].size
    leaves = []
    for _ in range(rounds):
        v, s, p, kind = tree.select(c_puct, fpu)
        logits, value = net(s, p, n_logits)
        tree.backup(v, s, p, kind, logits, value, None)
        leaves.append((v, kind))
    return tree, leaves


@pytest.mark.parametrize("version", ["barrage", "standard", "fives", "micro"])
def test_reference_invariants(version):
    """root N = rounds, N = 1 + the children's N on every expanded node, the root's children the expand action list,
    and a result that depends on nothing but its inputs"""
    t = traj(version)
    orc = logic(version)
    for i in _picks(t, 4):
        st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
        tree, leaves = _grow(orc, st, pl, 40, 400)
        a = tree.arrays()
        check_invariants(a, 40, 400)
        if a["first_child"][0] >= 0:
            f, n = a["first_child"][0], a["n_children"][0]
            assert np.array_equal(a["action"][f:f + n], action_list(orc, st, pl)), (version, i)
            assert abs(float(a["prior"][f:f + n].astype(np.float64).sum()) - 1) <= n * 2.0 ** -23
        else:
            assert data(st, OVER) or len(action_list(orc, st, pl)) == 0, (version, i)
        if data(st, OVER):
            assert all(k == LEAF_OVER and v == 0 for v, k in leaves)
        again = _grow(orc, st, pl, 40, 400)[0].arrays()
        assert all(np.array_equal(a[k], again[k]) for k in a if k != "used") and a["used"] == again["used"]


@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_small_pools_stop_growing_and_values_still_back_up(version):
    """a pool of the root's children + 1 nodes: the root expands once, nothing else does, and every round still adds
    one visit to the root"""
    t = traj(version)
    orc = logic(version)
    i = _picks(t, 2)[0]
    st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
    n = len(action_list(orc, st, pl))
    tree, _ = _grow(orc, st, pl, 30, 1 + n)
    a = tree.arrays()
    check_invariants(a, 30, 1 + n)
    assert a["used"] == 1 + n and np.all(a["first_child"][1:] == -1)
    one, leaves = _grow(orc, st, pl, 7, 1)
    assert one.arrays()["used"] == 1 and one.arrays()["visits"][0] == 7
    assert all(v == 0 and k == LEAF_EVAL for v, k in leaves)


def test_scores_are_float32_and_break_ties_low():
    """the score is float32 with one rounding per operation, fpu for unvisited children, and equal scores go to the
    lowest index"""
    f = np.float32
    s = scores([f(1.5), f(1.5), f(-2), f(0)], [3, 3, 5, 0], [f(0.25), f(0.25), f(0.5), f(0.125)], 11, 1, 1.25, -0.5)
    q0 = f(1.5) / f(3)
    u0 = ((f(1.25) * f(0.25)) * np.sqrt(f(11))) / f(4)
    u3 = ((f(1.25) * f(0.125)) * np.sqrt(f(11))) / f(1)
    assert s.dtype == np.float32 and s[0] == f(q0 + u0) and s[0] == s[1] and int(np.argmax(s)) == 0
    assert s[3] == f(f(-0.5) + u3)
    assert scores([f(2)], [4], [f(1)], 9, -1, 0.0, 0.0)[0] == f(-0.5)  # the mover's side: sigma = -1 flips W
    # u rounds (c_puct * P) first, then the product with sqrt(N_v), then the quotient
    c, p, r = f(1.1), f(0.3), np.sqrt(f(7))
    assert scores([f(0)], [0], [p], 7, 1, c, 0.0)[0] == f((c * p) * r)


def test_softmax_reference_edges():
    assert np.allclose(softmax64([-np.inf, -np.inf, -np.inf]), 1 / 3)
    p = softmax64([0.0, -np.inf, 0.0])
    assert p[1] == 0 and p[0] == p[2] == 0.5


# ---- the prior bound, on a numpy float32 emulation of the kernel's softmax ------------------------------------------
def _rounded(x, dtype):
    """float32 logits after rounding to dtype, as the kernel reads them"""
    return torch.from_numpy(np.ascontiguousarray(x)).to(dtype).float().numpy()


def _blocks(case, dtype, count, seed):
    """count child blocks of 1-120 legal logits of LOGIT_CASES case, rounded to dtype; a fifth of them with about 30 %
    of the entries at -inf"""
    rng = np.random.default_rng(seed)
    big = float(torch.finfo(dtype).max)
    for _ in range(count):
        n = int(rng.integers(1, 121))
        x = network_logits(rng, case, n, big)
        if case != "all_inf" and rng.random() < 0.2:
            hole = rng.random(n) < 0.3
            if not hole.all():
                x[hole] = -np.inf
        yield _rounded(x, dtype), rng


@pytest.mark.parametrize("case", LOGIT_CASES)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16], ids=["f32", "bf16", "f16"])
def test_prior_bound_holds_for_the_kernels_arithmetic(case, dtype):
    """float32 x - max, exp correctly rounded and then moved by up to 2 ulp (expf's error), a float32 sum and a float32
    division stay within prior_bound, and every block sums to 1 within n * 2^-23"""
    for x, rng in _blocks(case, dtype, 1500, 7):
        check_priors(softmax_f32(x, rng.uniform(-2, 2, x.size)), x)


def test_the_old_prior_bound_fails_on_ordinary_logits():
    """(n + 8) * 2^-24 relative, without the |x - max| term, fails on N(0, 10) logits even with exp correctly rounded:
    fl(x - max) alone is off by up to 2^-24 |x - max|, and exp keeps that as relative error.  prior_bound holds on the
    same blocks."""
    old = new = 0
    for x, _ in _blocks("sigma10", torch.float32, 2000, 11):
        p, w = softmax_f32(x).astype(np.float64), softmax64(x)
        ok = w >= 2.0 ** -126  # normal priors only: below them the old bound, having no absolute term, fails anyway
        old += bool(np.any((np.abs(p - w) > (x.size + 8) * 2.0 ** -24 * w) & ok))
        new += bool(np.any(np.abs(p - w) > prior_bound(x)))
    assert new == 0 and old >= 50, (old, new)  # 132 of the 2000 blocks break the old bound


def test_prior_bound_edges():
    """exact results the bound must allow: a single move, uniform -inf blocks, priors that underflow to 0"""
    one = softmax_f32([3.25])
    assert one[0] == 1 and prior_bound([3.25])[0] >= 2.0 ** -146
    for n in (1, 3, 7, 100):
        x = np.full(n, -np.inf, np.float32)
        p = softmax_f32(x)
        assert np.all(p == np.float32(1) / np.float32(n))
        check_priors(p, x)
    x = np.array([5, -107, -150, -np.inf], np.float32)
    p = softmax_f32(x)
    assert p[0] == 1 and np.all(p[1:] == 0)
    check_priors(p, x)
    big = np.finfo(np.float32).max
    x = np.array([big, -big, 0, big], np.float32)
    p = softmax_f32(x)
    assert p[0] == p[3] == 0.5 and p[1] == p[2] == 0
    check_priors(p, x)


# ---- argument checks without a device -------------------------------------------------------------------------------
def _tree(**null):
    from stratego_env_b200 import _lib
    names = [n for n, _ in _lib.SxGuidedTree._fields_]
    return _lib.SxGuidedTree(*(None if null.get(n) else 0x70000 + 0x1000 * k for k, n in enumerate(names)))


def _select(lib, cfg, st=None, num_envs=4, tree=None, max_nodes=64, c_puct=1.25, fpu=0.0, leaf=None, node=0x90000,
            kind=0xA0000):
    return lib.sx_guided_select(cfg, _fake_state(0x10000) if st is None else st, num_envs,
                                _tree() if tree is None else tree, max_nodes, c_puct, fpu,
                                _fake_state(0x20000) if leaf is None else leaf, node, kind, None)


def _backup(lib, cfg, leaf=None, num_envs=4, tree=None, max_nodes=64, node=0x90000, kind=0xA0000, logits=0xB0000,
            dtype=0, values=0xC0000):
    return lib.sx_guided_backup(cfg, _fake_state(0x20000) if leaf is None else leaf, num_envs,
                                _tree() if tree is None else tree, max_nodes, node, kind, logits, dtype, values, None)


TREE_FIELDS = ("visits", "value", "parent", "first_child", "n_children", "action", "prior", "used")


@pytest.mark.parametrize("case,kw,needle", [
    ("null config", {}, b"null config"),
    ("null state", {"st": "null"}, b"null state"),
    *[("null " + n, {"tree": n}, b"null tree") for n in TREE_FIELDS],
    ("null leaf states", {"leaf": "null"}, b"null leaf output"),
    ("null leaf node", {"node": None}, b"null leaf output"),
    ("null leaf kind", {"kind": None}, b"null leaf output"),
    ("leaf board is root board", {"leaf": "same"}, b"leaf_states.board is st.board"),
    ("zero max_nodes", {"max_nodes": 0}, b"max_nodes"),
    ("negative max_nodes", {"max_nodes": -5}, b"max_nodes"),
    ("negative c_puct", {"c_puct": -0.5}, b"c_puct"),
    ("nan c_puct", {"c_puct": math.nan}, b"c_puct"),
    ("inf c_puct", {"c_puct": math.inf}, b"c_puct"),
    ("nan fpu", {"fpu": math.nan}, b"fpu"),
    ("inf fpu", {"fpu": math.inf}, b"fpu"),
    ("-inf fpu", {"fpu": -math.inf}, b"fpu"),
])
def test_abi_select_refusals(case, kw, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        kw = dict(kw)
        if kw.get("st") == "null":
            kw["st"] = _lib.SxState()
        if kw.get("leaf") == "null":
            kw["leaf"] = _lib.SxState()
        elif kw.get("leaf") == "same":
            kw["leaf"] = _fake_state(0x10000)
        if "tree" in kw:
            kw["tree"] = _tree(**{kw["tree"]: True})
        assert _select(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


@pytest.mark.parametrize("case,kw,needle", [
    ("null config", {}, b"null config"),
    ("null leaf states", {"leaf": "null"}, b"null leaf state"),
    *[("null " + n, {"tree": n}, b"null tree") for n in TREE_FIELDS],
    ("null leaf node", {"node": None}, b"null leaf node"),
    ("null leaf kind", {"kind": None}, b"null leaf node or kind"),
    ("null logits", {"logits": None}, b"null logits"),
    ("null values", {"values": None}, b"null values"),
    ("zero max_nodes", {"max_nodes": 0}, b"max_nodes"),
    ("unknown dtype 3", {"dtype": 3}, b"unknown logits dtype"),
    ("unknown dtype -1", {"dtype": -1}, b"unknown logits dtype"),
])
def test_abi_backup_refusals(case, kw, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        kw = dict(kw)
        if kw.get("leaf") == "null":
            kw["leaf"] = _lib.SxState()
        if "tree" in kw:
            kw["tree"] = _tree(**{kw["tree"]: True})
        assert _backup(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_no_games_is_a_no_op():
    """num_envs <= 0 launches nothing (the fake pointers are never touched); the limits of every argument pass"""
    lib, cfg, keep = _config()
    try:
        for n in (0, -3):
            for nodes, c, fpu in ((1, 0.0, -3.0e38), ((1 << 31) - 1, 3.0e38, 3.0e38)):
                assert _select(lib, cfg, num_envs=n, max_nodes=nodes, c_puct=c, fpu=fpu) == 0, lib.sx_last_error()
            for dtype in (0, 1, 2):
                assert _backup(lib, cfg, num_envs=n, dtype=dtype) == 0, lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


# ---- the engine's checks, before any device is touched --------------------------------------------------------------
def _engine(monkeypatch):
    eng = _no_device_engine(monkeypatch)
    eng.layout.spatial_actions = 10 * 10 * 37
    eng.spatial_action_size = (10, 10, 37)
    return eng


def _host_tree(B=4, M=16, **change):
    """a guided SearchTree of host tensors (so that any use of it fails the device check)"""
    from stratego_env_b200.engine import SearchTree
    f = {n: torch.zeros(B, M, dtype=torch.float32 if n in ("value", "prior") else torch.int32)
         for n in ("visits", "value", "parent", "first_child", "n_children", "action", "prior")}
    f["used"] = torch.ones(B, dtype=torch.int32)
    f.update(change)
    return SearchTree(f["visits"], f["value"], f["parent"], f["first_child"], f["n_children"], f["action"],
                      used=f["used"], root_player=torch.ones(B, dtype=torch.int8), mask_shape=(10, 10, 37),
                      prior=f["prior"])


STATES = [None, "state", (1, 2, 3), _state()]
STATE_IDS = ["None", "str", "tuple", "host tensors"]


@pytest.mark.parametrize("state", STATES, ids=STATE_IDS)
def test_engine_rejects_bad_roots_before_touching_a_device(state, monkeypatch):
    eng = _engine(monkeypatch)
    with pytest.raises(ValueError, match="state"):
        eng.guided_tree(state, 16)
    with pytest.raises(ValueError, match="state"):
        eng.guided_select(state, _host_tree())


@pytest.mark.parametrize("max_nodes", [0, -1, True, 1.0, "7", None, 1 << 31])
def test_engine_rejects_bad_max_nodes_before_touching_a_device(max_nodes, monkeypatch):
    eng = _engine(monkeypatch)
    with pytest.raises(ValueError, match="max_nodes"):
        eng.guided_tree(_state(), max_nodes)


def _device_state_stub(monkeypatch, eng):
    """pretend the engine's state check passes, so that the tree, logits and value checks are reached"""
    monkeypatch.setattr(type(eng), "_check_state", lambda self, state: None)


@pytest.mark.parametrize("what", ["not a tree", "search tree", "int32 value", "short prior", "float used",
                                  "host tensors"])
def test_engine_rejects_bad_trees_before_touching_a_device(what, monkeypatch):
    eng = _engine(monkeypatch)
    _device_state_stub(monkeypatch, eng)
    tree = {"not a tree": "tree", "search tree": _host_tree(prior=None),
            "int32 value": _host_tree(value=torch.zeros(4, 16, dtype=torch.int32)),
            "short prior": _host_tree(prior=torch.zeros(4, 15)),
            "float used": _host_tree(used=torch.ones(4)), "host tensors": _host_tree()}[what]
    with pytest.raises(ValueError, match="tree"):
        eng.guided_select(_state(), tree)


@pytest.mark.parametrize("c_puct", [-0.1, math.nan, math.inf, -math.inf, 1e39, True, "1", None])
def test_engine_rejects_bad_c_puct_before_touching_a_device(c_puct, monkeypatch):
    eng = _engine(monkeypatch)
    _device_state_stub(monkeypatch, eng)
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    with pytest.raises(ValueError, match="c_puct"):
        eng.guided_select(_state(), _host_tree(), c_puct=c_puct)


@pytest.mark.parametrize("fpu", [math.nan, math.inf, -math.inf, 1e39, -1e39, True, "0", None])
def test_engine_rejects_bad_fpu_before_touching_a_device(fpu, monkeypatch):
    eng = _engine(monkeypatch)
    _device_state_stub(monkeypatch, eng)
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    with pytest.raises(ValueError, match="fpu"):
        eng.guided_select(_state(), _host_tree(), fpu=fpu)


def _leaves(B=4, **change):
    from stratego_env_b200.engine import Leaves
    f = dict(states=_state(B), node=torch.zeros(B, dtype=torch.int32), kind=torch.zeros(B, dtype=torch.int8))
    f.update(change)
    return Leaves(**f)


def _backup_args(**change):
    a = dict(tree=_host_tree(), leaves=_leaves(), logits=torch.zeros(4, 10, 10, 37), values=torch.zeros(4))
    a.update(change)
    return a


@pytest.mark.parametrize("what,kw,needle", [
    ("leaves not Leaves", dict(leaves=(1, 2, 3)), "leaves"),
    ("leaf states", dict(leaves=_leaves(states="x")), "state"),
    ("tree", dict(tree="tree"), "tree"),
    ("node dtype", dict(leaves=_leaves(node=torch.zeros(4, dtype=torch.int64))), "leaves.node"),
    ("kind shape", dict(leaves=_leaves(kind=torch.zeros(3, dtype=torch.int8))), "leaves.kind"),
    ("logits dtype", dict(logits=torch.zeros(4, 10, 10, 37, dtype=torch.float64)), "logits"),
    ("logits shape", dict(logits=torch.zeros(4, 10, 10, 36)), "logits"),
    ("logits rows", dict(logits=torch.zeros(5, 3700)), "logits"),
    ("logits not a tensor", dict(logits=np.zeros((4, 3700), np.float32)), "logits"),
    ("logits strided", dict(logits=torch.zeros(4, 7400)[:, ::2]), "logits"),
    ("values dtype", dict(values=torch.zeros(4, dtype=torch.float64)), "values"),
    ("values shape", dict(values=torch.zeros(4, 1)), "values"),
    ("values list", dict(values=[0.0] * 4), "values"),
])
def test_engine_rejects_bad_backup_arguments_before_touching_a_device(what, kw, needle, monkeypatch):
    eng = _engine(monkeypatch)
    args = _backup_args(**kw)
    if what not in ("leaf states",):
        _device_state_stub(monkeypatch, eng)
    if what not in ("tree", "leaves not Leaves"):
        monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    monkeypatch.setattr(eng, "device", torch.device("cpu"))  # host tensors pass the device test: the shape test fails
    with pytest.raises(ValueError, match=needle):
        eng.guided_backup(**args)
