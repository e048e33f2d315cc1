"""sx_guided_select_many / sx_guided_backup_many on the device: every round's L leaves per tree (node, kind, exported
state) and the whole tree against the reference of tests/_guided_batch_ref.py on recorded states of every variant,
with L from 1 to 64 and changing between rounds, virtual losses 0 to 2^24 and all three logit dtypes; L = 1 through the
new entry points against the one-leaf entry points byte for byte; the pending-visit buffer and what select leaves
alone; duplicate leaves, pools smaller than a round, OVER and STUCK leaves among the L; the batch split; no host
synchronisation; a full-size batch; the env forwarder."""
import numpy as np
import pytest
import torch

from _expand_ref import action_list, logic
from _golden import VERSIONS, traj
from _guided_batch_ref import BatchTree, check_invariants_many
from _guided_ref import LEAF_EVAL, LEAF_OVER, LEAF_STUCK, net
from test_expand_moves_gpu import _engine, _selfplay
from test_guided_search_gpu import STATE, TREE, _device_net, _host, _same, _tree_rows
from test_search_gpu import _recorded

pytestmark = pytest.mark.gpu


def _against_reference(e, version, dense, player, rows, Ls, max_nodes, c_puct=1.25, fpu=0.0, vl=1.0,
                       dtype=torch.float32):
    """grow trees from the imported states with rounds of Ls[r] leaves per tree; every round's leaves and the final
    trees against the reference (given the device's priors), the pending-visit buffer zero after every select; the
    count of each leaf kind"""
    orc = logic(version)
    B = len(player)
    st = e.import_ref_state(torch.as_tensor(dense, device="cuda"),
                            torch.as_tensor(np.asarray(player, np.int8), device="cuda"))
    tree = e.guided_tree(st, max_nodes)
    refs = [BatchTree(orc, dense[b], int(player[b]), max_nodes) for b in range(B)]
    n = e.layout.spatial_actions
    kinds = np.zeros(3, np.int64)
    for r, L in enumerate(Ls):
        leaves = e.guided_select(st, tree, c_puct=c_puct, fpu=fpu, leaves_per_tree=L, virtual_loss=vl)
        assert leaves.per_tree == L and leaves.node.shape == (B * L,)
        if tree.inflight is not None:
            assert int(tree.inflight.abs().sum()) == 0, (version, r)
        ld, lp = (x.cpu().numpy() for x in e.export_ref_state(leaves.states))
        node, kind = leaves.node.cpu().numpy(), leaves.kind.cpu().numpy()
        nets = [net(ld[i], int(lp[i]), n) for i in range(B * L)]
        logits = torch.as_tensor(np.stack([x for x, _ in nets])).to("cuda", dtype).view(B * L, *e.spatial_action_size)
        seen = logits.float().view(B * L, n).cpu().numpy()
        values = torch.as_tensor(np.array([v for _, v in nets], np.float32), device="cuda")
        e.guided_backup(tree, leaves, logits, values)
        prior = tree.prior.cpu().numpy()
        for b in range(B):
            want = refs[b].select_many(L, c_puct, fpu, vl)
            for j, (v, s, p, k) in enumerate(want):
                i = b * L + j
                what = (version, rows[b], r, L, j)
                assert (int(node[i]), int(kind[i])) == (v, k), (what, int(node[i]), int(kind[i]), v, k)
                assert np.array_equal(ld[i], s) and int(lp[i]) == p, what
                kinds[k] += 1
            refs[b].backup_many(want, seen[b * L:(b + 1) * L], [nets[b * L + j][1] for j in range(L)], prior[b])
    for b in range(B):
        want = refs[b].arrays()
        _same(_host(tree, b), want, (version, rows[b]))
        check_invariants_many(want, refs[b].ends, max_nodes)
        assert want["visits"][0] == sum(Ls)
    return st, tree, kinds


@pytest.mark.parametrize("version", VERSIONS)
def test_trees_and_leaves_equal_the_reference(version):
    """rounds of L = 1, 2, 7, 1, 4 on recorded states (both players to move): float32 logits with vl 1, bfloat16 with
    vl 0 and c_puct 0.5 / fpu -1, float16 with vl 3 and fpu -1"""
    e = _engine(version)
    dense, player, rows = _recorded(version)
    _against_reference(e, version, dense, player, rows, (1, 2, 7, 1, 4), 2000)
    h = len(rows) // 2
    pick = [0, 1, h, h + 1, len(rows) - 1]
    sub = (dense[pick], player[pick], [rows[i] for i in pick])
    _against_reference(e, version, *sub, (1, 5, 3, 8), 2000, c_puct=0.5, fpu=-1.0, vl=0.0, dtype=torch.bfloat16)
    _against_reference(e, version, *sub, (3, 1, 6, 2), 2000, fpu=-1.0, vl=3.0, dtype=torch.float16)


@pytest.mark.parametrize("L", [1, 2, 7, 32, 33, 64])
@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_leaves_per_tree(version, L):
    """an L = 1 round, then two rounds of L (32 and 33 straddle a warp, 64 two); on micro the rounds hold OVER leaves
    among the EVAL ones"""
    e = _engine(version)
    dense, player, rows = _recorded(version)
    _, _, kinds = _against_reference(e, version, dense, player, rows, (1, L, L), 3000)
    if version == "micro" and L >= 32:
        assert kinds[LEAF_OVER] > 0 and kinds[LEAF_EVAL] > 0, kinds


@pytest.mark.parametrize("vl", [0.0, 1.0, 3.0, 2.0 ** 24])
def test_virtual_loss(vl):
    e = _engine("barrage")
    dense, player, rows = _recorded("barrage")
    _against_reference(e, "barrage", dense, player, rows, (1, 8, 16, 8), 2000, vl=vl)


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_pools_smaller_than_a_round(version):
    """pools of 1, 2, the first root's children plus one, and 70 nodes with rounds of 8 and 33 leaves: duplicate leaves
    at unexpanded nodes, a pool that fills between two leaves of a round, values that still back up"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 3)
    n_root = len(action_list(logic(version), dense[0], player[0]))
    for nodes in (1, 2, n_root + 1, 70):
        _, tree, _ = _against_reference(e, version, dense, player, rows, (8, 1, 33, 8), nodes)
        assert bool((tree.used <= nodes).all()) and bool((tree.visits[:, 0] == 50).all())


@pytest.mark.parametrize("version,row", [("barrage", 237), ("micro", 36), ("tiny", 181)])
def test_stuck_and_finished_roots(version, row):
    """a stuck root and finished roots give L STUCK / OVER leaves per round, stay used = 1 and back up every one"""
    e = _engine(version)
    t = traj(version)
    over = [i for i in range(t["states"].shape[0]) if t["states"][i][5][0, 1]][:2]
    dense = t["states"][[row] + over].astype(np.int64)
    player = np.array([-int(t["players"][row])] + [int(t["players"][i]) for i in over], np.int64)
    _, tree, kinds = _against_reference(e, version, dense, player, [row] + over, (1, 4, 9), 50)
    assert kinds[LEAF_STUCK] == 14 and kinds[LEAF_OVER] == 14 * len(over) and kinds[LEAF_EVAL] == 0
    assert bool((tree.used == 1).all()) and bool((tree.visits[:, 0] == 14).all())
    assert float(tree.value[0, 0]) == 14.0 * -int(player[0])


def test_first_round_of_an_empty_tree():
    """every leaf of the first round of an empty tree is the root; the root is expanded once and gains N = L"""
    e = _engine("barrage")
    st = _selfplay(e, 256, 60, seed=6)
    tree = e.guided_tree(st, 600)
    leaves = e.guided_select(st, tree, leaves_per_tree=8)
    assert bool((leaves.node == 0).all())
    eval_root = (leaves.kind.view(256, 8)[:, 0] == LEAF_EVAL)
    logits, values = _device_net(e, leaves)
    e.guided_backup(tree, leaves, logits, values)
    off = e.expand_moves(st).offsets
    n_root = (off[1:] - off[:-1]).to(torch.int32)
    assert bool((tree.visits[:, 0] == 8).all())
    assert torch.equal(tree.used[eval_root], 1 + n_root[eval_root])
    assert torch.equal(tree.n_children[:, 0][eval_root], n_root[eval_root])


def _old_abi_round(e, st, tree, c_puct, fpu, logits_of):
    """one round through sx_guided_select / sx_guided_backup, the one-leaf entry points"""
    from stratego_env_b200 import _lib
    from stratego_env_b200.engine import Leaves, _stream
    B, M = st.num_envs, tree.visits.shape[1]
    leaves = Leaves(e.alloc_state(B), torch.empty(B, dtype=torch.int32, device="cuda"),
                    torch.empty(B, dtype=torch.int8, device="cuda"))
    _lib.check(e.lib.sx_guided_select(e._cfg, st.as_struct(), B, e._guided_struct(tree), M, float(c_puct), float(fpu),
                                      leaves.states.as_struct(), leaves.node.data_ptr(), leaves.kind.data_ptr(),
                                      _stream()), "sx_guided_select")
    logits, values = logits_of(leaves)
    _lib.check(e.lib.sx_guided_backup(e._cfg, leaves.states.as_struct(), B, e._guided_struct(tree), M,
                                      leaves.node.data_ptr(), leaves.kind.data_ptr(), logits.data_ptr(), 0,
                                      values.data_ptr(), _stream()), "sx_guided_backup")
    return leaves


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_one_leaf_through_the_new_entry_points_is_the_one_leaf_search(version):
    """L = 1 through guided_select / guided_backup (sx_guided_select_many / sx_guided_backup_many) and through
    sx_guided_select / sx_guided_backup: the same leaves every round and the same trees, byte for byte (every column,
    unused ones included, from trees that start byte-identical)"""
    e = _engine(version)
    st = _selfplay(e, 512, 60, seed=9)
    a, b = e.guided_tree(st, 700), e.guided_tree(st, 700)
    for k in TREE:
        getattr(a, k).zero_()
        getattr(b, k).zero_()
    for x in (a, b):
        for t, v in ((x.parent, -1), (x.first_child, -1), (x.action, -1), (x.prior, 1.0)):
            t[:, 0].fill_(v)
        x.used.fill_(1)
    for r in range(12):
        c_puct, fpu = (1.25, 0.0) if r % 2 else (0.7, -0.5)
        old = _old_abi_round(e, st, a, c_puct, fpu, lambda lv: _device_net(e, lv))
        new = e.guided_select(st, b, c_puct=c_puct, fpu=fpu, virtual_loss=3.0)
        assert new.per_tree == 1 and b.inflight is None
        for n in STATE:
            assert torch.equal(getattr(old.states, n), getattr(new.states, n)), (r, n)
        assert torch.equal(old.node, new.node) and torch.equal(old.kind, new.kind), r
        e.guided_backup(b, new, *_device_net(e, new))
        for k in TREE:
            assert torch.equal(_bits(getattr(a, k)), _bits(getattr(b, k))), (r, k)


def test_select_leaves_the_tree_and_the_buffer_alone():
    """after rounds of mixed L: two selects of 8 leaves without a backup leave every tree field byte-identical and the
    pending-visit buffer all zero, and return the same leaves"""
    e = _engine("barrage")
    st = _selfplay(e, 512, 60, seed=4)
    before = st.clone()
    tree = e.guided_tree(st, 900)
    for L in (1, 4, 8, 2):
        leaves = e.guided_select(st, tree, leaves_per_tree=L)
        e.guided_backup(tree, leaves, *_device_net(e, leaves))
    snap = {k: _bits(getattr(tree, k)).clone() for k in TREE}
    x = e.guided_select(st, tree, c_puct=0.8, fpu=-0.25, leaves_per_tree=8, virtual_loss=2.0)
    assert int(tree.inflight.abs().sum()) == 0
    y = e.guided_select(st, tree, c_puct=0.8, fpu=-0.25, leaves_per_tree=8, virtual_loss=2.0)
    assert int(tree.inflight.abs().sum()) == 0
    for k in TREE:
        assert torch.equal(_bits(getattr(tree, k)), snap[k]), k
    for n in STATE:
        assert torch.equal(getattr(st, n), getattr(before, n)), n
        assert torch.equal(getattr(x.states, n), getattr(y.states, n)), n
    assert torch.equal(x.node, y.node) and torch.equal(x.kind, y.kind)
    # the pending visits spread a tree's leaves over several nodes
    distinct = lambda lv: sum(len(set(r)) for r in lv.node.view(512, 8).tolist())  # noqa: E731
    assert distinct(x) > 512


def _rounds(e, st, tree, Ls, vl=1.0):
    for L in Ls:
        leaves = e.guided_select(st, tree, leaves_per_tree=L, virtual_loss=vl)
        e.guided_backup(tree, leaves, *_device_net(e, leaves))
    return tree


def test_deterministic_and_independent_of_the_batch_split():
    """two runs give identical trees; rows [lo, hi) grown alone equal those rows"""
    e = _engine("barrage")
    st = _selfplay(e, 300, 80, seed=2)
    Ls = (1, 4, 8, 3, 16, 1, 8)
    x = _tree_rows(_rounds(e, st, e.guided_tree(st, 1200), Ls))
    y = _tree_rows(_rounds(e, st, e.guided_tree(st, 1200), Ls))
    for k in TREE:
        assert torch.equal(x[k], y[k]), k
    lo, hi = 70, 211
    part = st.select(lo, hi)
    part = type(part)(*(getattr(part, n).contiguous() for n in STATE))
    z = _tree_rows(_rounds(e, part, e.guided_tree(part, 1200), Ls))
    for k in TREE:
        assert torch.equal(z[k], x[k][lo:hi]), k


def test_a_round_of_several_leaves_does_not_synchronise_the_host():
    """after one warm-up round (which allocates the pending-visit buffer), rounds of L > 1 never synchronise"""
    e = _engine("barrage")
    st = _selfplay(e, 256, 40, seed=5)
    tree = e.guided_tree(st, 800)
    _rounds(e, st, tree, (1, 8))
    leaves = e.guided_select(st, tree, leaves_per_tree=8)
    logits, values = _device_net(e, leaves)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for vl in (1.0, 0.0):
            leaves = e.guided_select(st, tree, leaves_per_tree=8, virtual_loss=vl)
            e.guided_backup(tree, leaves, logits, values)
        leaves = e.guided_select(st, tree, c_puct=0.5, fpu=-1.0, leaves_per_tree=8)
        e.guided_backup(tree, leaves, logits.to(torch.bfloat16), values)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert bool((tree.visits[:, 0] == 1 + 8 * 4).all())


def _device_invariants(tree, ends):
    """the contract's consequences on every tree, with torch ops; ends int64 [B, M]: selections that ended at each node"""
    B, M = tree.visits.shape
    used = tree.used.long()
    cols = torch.arange(M, device="cuda")[None, :]
    live = cols < used[:, None]
    assert bool((used >= 1).all()) and bool((used <= M).all())
    assert bool((tree.visits[:, 0].long() == ends.sum(1)).all()) and bool((tree.parent[:, 0] == -1).all())
    N = torch.where(live, tree.visits, 0).long()
    par = tree.parent.long()
    child = live & (cols > 0)
    assert bool(((par >= 0) & (par < cols))[child].all())
    slot = torch.where(child, par, M)
    kid_sum = torch.zeros(B, M + 1, dtype=torch.long, device="cuda").scatter_add_(1, slot, N)[:, :M]
    kid_n = torch.zeros(B, M + 1, dtype=torch.long, device="cuda").scatter_add_(1, slot, child.long())[:, :M]
    fc, nc = tree.first_child.long(), tree.n_children.long()
    expanded = live & (fc >= 0)
    assert bool((N == ends + kid_sum)[live].all())
    assert bool((nc == kid_n)[live].all())
    assert bool(((fc + nc <= used[:, None]) & (fc > cols))[expanded].all())
    W = torch.where(live, tree.value, 0.0)
    assert bool((W.abs() <= N.float())[live].all())
    assert int(tree.inflight.abs().sum()) == 0


def test_full_size_barrage():
    """65 536 de-phased Barrage trees: one L = 1 round, then 15 rounds of L = 8 with the device evaluator; the invariants
    on every tree and the reference on sampled rows, given the logits and values the device evaluator gave them"""
    e = _engine("barrage")
    B, M, L = 65536, 2048, 8
    Ls = (1,) + (L,) * 15
    st = _selfplay(e, B, 200, seed=8)
    rows = (0, 1, 777, 40000, 65535)
    record = {b: [] for b in rows}
    tree = e.guided_tree(st, M)
    ends = torch.zeros(B, M, dtype=torch.long, device="cuda")
    for Lr in Ls:
        leaves = e.guided_select(st, tree, leaves_per_tree=Lr)
        logits, values = _device_net(e, leaves)
        ends.view(-1).scatter_add_(0, (torch.arange(B, device="cuda").repeat_interleave(Lr) * M
                                       + leaves.node.long()), torch.ones(B * Lr, dtype=torch.long, device="cuda"))
        for b in rows:
            record[b].append((Lr, logits[b * Lr:(b + 1) * Lr].reshape(Lr, -1).cpu().numpy(),
                              values[b * Lr:(b + 1) * Lr].cpu().numpy()))
        e.guided_backup(tree, leaves, logits, values)
        del logits, values, leaves
    _device_invariants(tree, ends)
    dense, player = (x.cpu().numpy() for x in e.export_ref_state(st))
    orc = logic("barrage")
    prior = tree.prior[list(rows)].cpu().numpy()
    for i, b in enumerate(rows):
        ref = BatchTree(orc, dense[b], int(player[b]), M)
        for Lr, logits, values in record[b]:
            ref.backup_many(ref.select_many(Lr, 1.25, 0.0, 1.0), logits, values, prior[i])
        _same(_host(tree, b), ref.arrays(), b)


def test_batched_env_forwards_its_games():
    from stratego_env_b200.batched_env import BatchedStrategoEnv
    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=64, device="cuda:0", seed=3, env_base=1000)
    env.reset()
    e = env.engine
    tree, want = env.guided_tree(300), e.guided_tree(env.state, 300)
    for L in (1, 4, 4, 2):
        leaves = env.guided_select(tree, c_puct=0.9, leaves_per_tree=L, virtual_loss=0.5)
        ref = e.guided_select(env.state, want, c_puct=0.9, leaves_per_tree=L, virtual_loss=0.5)
        assert leaves.per_tree == L and torch.equal(leaves.node, ref.node) and torch.equal(leaves.kind, ref.kind)
        for n in STATE:
            assert torch.equal(getattr(leaves.states, n), getattr(ref.states, n)), n
        logits, values = _device_net(e, leaves)
        e.guided_backup(tree, leaves, logits, values)
        e.guided_backup(want, ref, logits, values)
    x, y = _tree_rows(tree), _tree_rows(want)
    for k in TREE:
        assert torch.equal(x[k], y[k]), k
    visits, _ = tree.root_stats()
    assert int(visits.sum()) == 64 * 10  # 11 leaves per tree, the first of them the root itself
