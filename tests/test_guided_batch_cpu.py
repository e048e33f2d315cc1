"""No-GPU checks of guided search with several leaves per tree (sx_guided_select_many / sx_guided_backup_many): the
reference of tests/_guided_batch_ref.py at one leaf per round against _guided_ref.GuidedTree, the virtual-visit score at
V = 0 against the one-leaf score, the contract's consequences over rounds of mixed L, and the argument checks of the C
ABI and of StrategoEngine.guided_select / guided_backup before any device is touched."""
import math

import numpy as np
import pytest
import torch

from _expand_ref import action_list, logic
from _golden import traj
from _guided_batch_ref import BatchTree, check_invariants_many, scores_vl
from _guided_ref import LEAF_EVAL, GuidedTree, net, scores
from test_expand_moves_cpu import _config, _fake_state, _no_device_engine, _state

f32 = np.float32


def _picks(t, k):
    """k recorded states spread over the trajectory, the first of them a game start"""
    n = t["states"].shape[0]
    return sorted({int(np.flatnonzero(t["game_start"])[0]), *np.linspace(0, n - 1, k).astype(int).tolist()})


def _round(tree, L, n_logits, c_puct=1.25, fpu=0.0, vl=1.0):
    """one round of L leaves with the test network; the leaves"""
    leaves = tree.select_many(L, c_puct, fpu, vl)
    nets = [net(s, p, n_logits) for _, s, p, _ in leaves]
    tree.backup_many(leaves, [x for x, _ in nets], [z for _, z in nets], None)
    return leaves


@pytest.mark.parametrize("version", ["barrage", "standard", "fives", "micro"])
@pytest.mark.parametrize("vl", [0.0, 1.0, 3.0])
def test_one_leaf_per_round_is_the_one_leaf_reference(version, vl):
    """L = 1: every round's leaf and the final tree equal GuidedTree's, whatever the virtual loss"""
    t = traj(version)
    orc = logic(version)
    for i in _picks(t, 3):
        st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
        n_logits = orc.current_obs(st, pl, obs_mode=0)[0].size
        old, new = GuidedTree(orc, st, pl, 300), BatchTree(orc, st, pl, 300)
        for r in range(30):
            v, s, p, k = old.select(1.25, -0.25)
            logits, value = net(s, p, n_logits)
            old.backup(v, s, p, k, logits, value, None)
            (lv, ls, lp, lk), = _round(new, 1, n_logits, 1.25, -0.25, vl)
            assert (lv, lk, lp) == (v, k, p) and np.array_equal(ls, s), (version, i, r)
        a, b = old.arrays(), new.arrays()
        assert a["used"] == b["used"]
        for k in a:
            if k != "used":
                assert np.array_equal(np.asarray(a[k]).view(np.int32) if a[k].dtype == f32 else a[k],
                                      np.asarray(b[k]).view(np.int32) if b[k].dtype == f32 else b[k]), k


def _bits(x):
    return np.asarray(x, f32).view(np.int32)


@pytest.mark.parametrize("vl", [0.0, 1.0, 3.0, 2.0 ** 24])
def test_the_virtual_visit_score_at_no_pending_visit_is_the_one_leaf_score(vl):
    """V = 0: vl * 0 = +0 and sigma * W - (+0) = sigma * W, so every score is bit for bit the one-leaf score, -0
    included, for either mover, visited or not, and at the float32 extremes"""
    rng = np.random.default_rng(3)
    n = 4000
    W = (rng.standard_normal(n) * 8).astype(f32)
    W[::7], W[1::7] = f32(0.0), f32(-0.0)
    N = rng.integers(0, 60, n)
    N[::5] = 0
    W[N == 0] = 0
    P = rng.random(n).astype(f32)
    P[::11] = 0
    for sigma in (1, -1):
        for n_parent, c_puct, fpu in ((37, 1.25, 0.0), (1, 0.0, -0.0), (0, 1.25, -1.0), ((1 << 24) - 1, 3.0e38, 3.0e38)):
            with np.errstate(over="ignore"):
                old = scores(W, N, P, n_parent, sigma, c_puct, fpu)
            new = scores_vl(W, N, np.zeros(n, np.int64), P, n_parent, 0, sigma, c_puct, fpu, vl)
            assert np.array_equal(_bits(old), _bits(new)), (sigma, n_parent, c_puct, fpu)
    # -0 survives: sigma * W = -0, q = -0 / 3 = -0, and a prior of -0 gives u = -0, so the score is -0
    assert _bits(scores_vl([f32(0)], [3], [0], [f32(-0.0)], 3, 0, -1, 1.0, 0.0, vl))[0] == _bits(f32(-0.0))
    assert _bits(scores([f32(0)], [3], [f32(-0.0)], 3, -1, 1.0, 0.0))[0] == _bits(f32(-0.0))


def test_the_virtual_visit_score():
    """each pending visit counts in n and in the parent's count, and takes vl from the mover's value; a child reached
    only by pending visits has q = -vl"""
    s = scores_vl([f32(1.5), f32(0)], [3, 0], [2, 1], [f32(0.25), f32(0.5)], 9, 3, 1, 1.25, -0.5, 3.0)
    r = np.sqrt(f32(12))
    assert s[0] == f32((f32(1.5) - f32(6)) / f32(5) + ((f32(1.25) * f32(0.25)) * r) / f32(6))
    assert s[1] == f32(f32(-3) + ((f32(1.25) * f32(0.5)) * r) / f32(2))
    assert scores_vl([f32(2)], [4], [1], [f32(1)], 9, 1, -1, 0.0, 0.0, 0.0)[0] == f32(-2) / f32(5)  # vl = 0: visits


def _expanded_once(tree):
    """no node has children twice: children blocks are disjoint and every one was made for its parent"""
    a = tree.arrays()
    fc, nc = np.asarray(a["first_child"]), np.asarray(a["n_children"])
    blocks = sorted((f, f + n) for f, n in zip(fc, nc) if f >= 0)
    assert all(b[0] >= c[1] for c, b in zip(blocks, blocks[1:]))
    assert sum(n for _, n in ((f, e - f) for f, e in blocks)) == a["used"] - 1 or a["used"] == 1


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_invariants_over_rounds_of_mixed_leaves_per_tree(version):
    """rounds of L = 1, 4, 7, 2, 32, 1, 8, 33: root N = the leaves backed up, N = e + the children's N everywhere, every
    node expanded once; the first round of an empty tree with L > 1 gives L root leaves and one expansion"""
    t = traj(version)
    orc = logic(version)
    Ls = (1, 4, 7, 2, 32, 1, 8, 33)
    for i in _picks(t, 2):
        st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
        n_logits = orc.current_obs(st, pl, obs_mode=0)[0].size
        tree = BatchTree(orc, st, pl, 2000)
        for L in Ls:
            _round(tree, L, n_logits, vl=1.0)
        a = tree.arrays()
        check_invariants_many(a, tree.ends, 2000)
        assert a["visits"][0] == sum(Ls)
        _expanded_once(tree)
        again = BatchTree(orc, st, pl, 2000)
        for L in Ls:
            _round(again, L, n_logits, vl=1.0)
        b = again.arrays()
        assert all(np.array_equal(a[k], b[k]) for k in a if k != "used") and a["used"] == b["used"]
        first = BatchTree(orc, st, pl, 2000)
        leaves = _round(first, 5, n_logits)
        if leaves[0][3] == LEAF_EVAL:
            assert all(v == 0 for v, _, _, _ in leaves)
            assert first.arrays()["visits"][0] == 5 and first.used == 1 + len(action_list(orc, st, pl))


def test_virtual_loss_spreads_the_leaves():
    """after an L = 1 round expands the root, a round of L <= the root's children with vl = 1 and fpu = 0 puts no two
    leaves on the same child while unvisited children remain (a pending visit makes q = -1 < fpu)"""
    t = traj("barrage")
    orc = logic("barrage")
    i = _picks(t, 2)[0]
    st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
    n_logits = orc.current_obs(st, pl, obs_mode=0)[0].size
    tree = BatchTree(orc, st, pl, 4000)
    _round(tree, 1, n_logits)
    n = tree.t["n_children"][0]
    L = min(n, 8)
    leaves = tree.select_many(L, 0.0, 0.0, 1.0)  # c_puct = 0: q alone decides
    assert len({v for v, _, _, _ in leaves}) == L


def test_a_pool_that_fills_in_the_middle_of_a_round():
    """a pool with room for the root's children and a few more: expansions stop at the first leaf that does not fit,
    later leaves of the round still back up, and the invariants hold"""
    t = traj("barrage")
    orc = logic("barrage")
    i = _picks(t, 2)[0]
    st, pl = t["states"][i].astype(np.int64), int(t["players"][i])
    n_logits = orc.current_obs(st, pl, obs_mode=0)[0].size
    n = len(action_list(orc, st, pl))
    M = 1 + n + n // 2
    tree = BatchTree(orc, st, pl, M)
    _round(tree, 1, n_logits)
    for L in (8, 8, 8):
        _round(tree, L, n_logits, fpu=-0.5)
    a = tree.arrays()
    check_invariants_many(a, tree.ends, M)
    assert a["visits"][0] == 25 and a["used"] <= M


# ---- argument checks without a device -------------------------------------------------------------------------------
def _tree(**null):
    from stratego_env_b200 import _lib
    names = [n for n, _ in _lib.SxGuidedTree._fields_]
    return _lib.SxGuidedTree(*(None if null.get(n) else 0x70000 + 0x1000 * k for k, n in enumerate(names)))


def _select_many(lib, cfg, st=None, num_envs=4, tree=None, max_nodes=64, c_puct=1.25, fpu=0.0, L=2, vl=1.0,
                 inflight=0xD0000, leaf=None, node=0x90000, kind=0xA0000):
    return lib.sx_guided_select_many(cfg, _fake_state(0x10000) if st is None else st, num_envs,
                                     _tree() if tree is None else tree, max_nodes, c_puct, fpu, L, vl, inflight,
                                     _fake_state(0x20000) if leaf is None else leaf, node, kind, None)


def _backup_many(lib, cfg, leaf=None, num_envs=4, tree=None, max_nodes=64, L=2, node=0x90000, kind=0xA0000,
                 logits=0xB0000, dtype=0, values=0xC0000):
    return lib.sx_guided_backup_many(cfg, _fake_state(0x20000) if leaf is None else leaf, num_envs,
                                     _tree() if tree is None else tree, max_nodes, L, node, kind, logits, dtype, values,
                                     None)


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
    ("negative c_puct", {"c_puct": -0.5}, b"c_puct"),
    ("nan c_puct", {"c_puct": math.nan}, b"c_puct"),
    ("inf fpu", {"fpu": math.inf}, b"fpu"),
    ("zero L", {"L": 0}, b"leaves_per_tree"),
    ("negative L", {"L": -3}, b"leaves_per_tree"),
    ("L 1025", {"L": 1025}, b"leaves_per_tree"),
    ("negative vl", {"vl": -1.0}, b"virtual_loss"),
    ("tiny negative vl", {"vl": -1e-30}, b"virtual_loss"),
    ("nan vl", {"vl": math.nan}, b"virtual_loss"),
    ("inf vl", {"vl": math.inf}, b"virtual_loss"),
    ("vl above 2^24", {"vl": 16777218.0}, b"virtual_loss"),
    ("null inflight with L 2", {"inflight": None}, b"inflight"),
    ("null inflight with L 1024", {"inflight": None, "L": 1024}, b"inflight"),
])
def test_abi_select_many_refusals(case, kw, needle):
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
        assert _select_many(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error() and b"sx_guided_select_many" in lib.sx_last_error()
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
    ("zero L", {"L": 0}, b"leaves_per_tree"),
    ("L 1025", {"L": 1025}, b"leaves_per_tree"),
])
def test_abi_backup_many_refusals(case, kw, needle):
    from stratego_env_b200 import _lib
    lib, cfg, keep = _config()
    try:
        kw = dict(kw)
        if kw.get("leaf") == "null":
            kw["leaf"] = _lib.SxState()
        if "tree" in kw:
            kw["tree"] = _tree(**{kw["tree"]: True})
        assert _backup_many(lib, None if case == "null config" else cfg, **kw) != 0
        assert needle in lib.sx_last_error() and b"sx_guided_backup_many" in lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


def test_abi_limits_pass_and_no_trees_is_a_no_op():
    """num_envs <= 0 launches nothing (the fake pointers are never touched) once every argument passes: L of 1 and
    1024, vl of 0, -0 and 2^24, a null inflight buffer with L = 1"""
    lib, cfg, keep = _config()
    try:
        for n in (0, -3):
            for L, vl, inflight in ((1, 0.0, None), (1, 2.0 ** 24, 0xD0000), (1024, -0.0, 0xD0000), (7, 1.0, 0xD0000)):
                assert _select_many(lib, cfg, num_envs=n, L=L, vl=vl, inflight=inflight) == 0, lib.sx_last_error()
                assert _backup_many(lib, cfg, num_envs=n, L=L) == 0, lib.sx_last_error()
    finally:
        lib.sx_config_destroy(cfg)


# ---- the engine's checks, before any device is touched --------------------------------------------------------------
def _engine(monkeypatch):
    eng = _no_device_engine(monkeypatch)
    eng.layout.spatial_actions = 10 * 10 * 37
    eng.spatial_action_size = (10, 10, 37)
    monkeypatch.setattr(type(eng), "_check_state", lambda self, state: None)
    return eng


def _host_tree(B=4, M=16, **change):
    """a guided SearchTree of host tensors"""
    from stratego_env_b200.engine import SearchTree
    f = {n: torch.zeros(B, M, dtype=torch.float32 if n in ("value", "prior") else torch.int32)
         for n in ("visits", "value", "parent", "first_child", "n_children", "action", "prior")}
    f["used"] = torch.ones(B, dtype=torch.int32)
    f.update(change)
    return SearchTree(f["visits"], f["value"], f["parent"], f["first_child"], f["n_children"], f["action"],
                      used=f["used"], root_player=torch.ones(B, dtype=torch.int8), mask_shape=(10, 10, 37),
                      prior=f["prior"], inflight=f.get("inflight"))


@pytest.mark.parametrize("L", [0, -1, 1025, True, 2.0, "2", None])
def test_engine_rejects_bad_leaves_per_tree_before_touching_a_device(L, monkeypatch):
    eng = _engine(monkeypatch)
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    with pytest.raises(ValueError, match="leaves_per_tree"):
        eng.guided_select(_state(), _host_tree(), leaves_per_tree=L)


@pytest.mark.parametrize("vl", [-1.0, -1e-30, math.nan, math.inf, 2.0 ** 24 + 2, 1e39, True, "1", None])
def test_engine_rejects_bad_virtual_loss_before_touching_a_device(vl, monkeypatch):
    eng = _engine(monkeypatch)
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    with pytest.raises(ValueError, match="virtual_loss"):
        eng.guided_select(_state(), _host_tree(), leaves_per_tree=2, virtual_loss=vl)


@pytest.mark.parametrize("what", ["int64", "short", "strided", "host", "list"])
@pytest.mark.parametrize("L", [1, 4])
def test_engine_rejects_a_bad_inflight_buffer_before_touching_a_device(what, L, monkeypatch):
    """a tree's inflight buffer, when present, is checked at every L"""
    eng = _engine(monkeypatch)
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: 16)
    bad = {"int64": torch.zeros(4, 16, dtype=torch.int64), "short": torch.zeros(4, 15, dtype=torch.int32),
           "strided": torch.zeros(4, 32, dtype=torch.int32)[:, ::2], "host": torch.zeros(4, 16, dtype=torch.int32),
           "list": [0] * 64}[what]
    with pytest.raises(ValueError, match="inflight"):
        eng.guided_select(_state(), _host_tree(inflight=bad), leaves_per_tree=L)


def _leaves(rows=8, per_tree=2, **change):
    from stratego_env_b200.engine import Leaves
    f = dict(states=_state(rows), node=torch.zeros(rows, dtype=torch.int32), kind=torch.zeros(rows, dtype=torch.int8),
             per_tree=per_tree)
    f.update(change)
    return Leaves(**f)


@pytest.mark.parametrize("what,kw,needle", [
    ("per_tree 0", dict(leaves=_leaves(per_tree=0)), "per_tree"),
    ("per_tree 1025", dict(leaves=_leaves(per_tree=1025)), "per_tree"),
    ("per_tree float", dict(leaves=_leaves(per_tree=2.0)), "per_tree"),
    ("rows not a multiple", dict(leaves=_leaves(rows=7, per_tree=2)), "multiple"),
    ("node rows of the trees", dict(leaves=_leaves(node=torch.zeros(4, dtype=torch.int32))), "leaves.node"),
    ("logits rows of the trees", dict(logits=torch.zeros(4, 10, 10, 37)), "logits"),
    ("values rows of the trees", dict(values=torch.zeros(4)), "values"),
])
def test_engine_rejects_bad_many_leaf_backups_before_touching_a_device(what, kw, needle, monkeypatch):
    """leaves of L per tree: B * L rows in leaves, logits and values, B trees"""
    eng = _engine(monkeypatch)
    seen = []
    monkeypatch.setattr(type(eng), "_check_guided_tree", lambda self, tree, B: seen.append(B) or 16)
    monkeypatch.setattr(eng, "device", torch.device("cpu"))  # host tensors pass the device test: the shape test fails
    args = dict(tree=_host_tree(), leaves=_leaves(), logits=torch.zeros(8, 10, 10, 37), values=torch.zeros(8))
    args.update(kw)
    with pytest.raises(ValueError, match=needle):
        eng.guided_backup(**args)
    assert seen in ([], [4])  # the trees are B = rows / L


def test_the_float_check_refuses_what_float32_cannot_hold():
    """the engine's float check (c_puct, fpu, virtual_loss) takes a Python float without numpy; it refuses exactly the
    values that round to +-inf or NaN in float32, as numpy's conversion does for every other type"""
    from stratego_env_b200.engine import StrategoEngine

    def passes(v):
        try:
            StrategoEngine._check_float("x", v)
            return True
        except ValueError:
            return False
    t = 3.4028235677973366e38  # 2^128 - 2^103: float32 rounds it (a tie, to even) to inf
    rng = np.random.default_rng(5)
    near = [*rng.uniform(3.40282346e38, 3.40282358e38, 500), math.nextafter(t, 0), t, math.nextafter(t, math.inf)]
    for v in near + [0.0, -0.0, 1.0, 1e-300, math.inf, math.nan]:
        for x in (v, -v):
            with np.errstate(over="ignore"):
                want = bool(np.isfinite(np.float32(x)))
            assert passes(x) == want and passes(np.float64(x)) == want, x
