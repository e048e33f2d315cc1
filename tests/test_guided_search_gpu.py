"""sx_guided_select / sx_guided_backup on the device: every round's leaves (node, kind, exported state) and the whole tree
(seven node fields and used) against the reference of tests/_guided_ref.py on recorded states of every variant, with
float32, bfloat16 and float16 logits; finished and stuck roots; pool exhaustion; the root's children against
expand_moves; what select leaves alone; determinism and the batch split; no host synchronisation; a full-size batch
with an evaluator on the device; the env forwarders.  _against_reference also serves
tests/test_guided_search_edges_gpu.py, which brings its own networks."""
import numpy as np
import pytest
import torch

from _expand_ref import action_list, logic
from _golden import VERSIONS, traj
from _guided_ref import FIELDS, LEAF_EVAL, LEAF_OVER, LEAF_STUCK, GuidedTree, check_invariants, net
from test_expand_moves_gpu import _engine, _selfplay
from test_search_gpu import _recorded

pytestmark = pytest.mark.gpu

STATE = ("board", "aux", "captured")
TREE = ("visits", "value", "parent", "first_child", "n_children", "action", "prior", "used")


def _host(tree, b):
    """tree b as the reference's arrays(): the used columns of every field"""
    used = int(tree.used[b])
    out = {k: getattr(tree, k)[b, :used].cpu().numpy() for k in FIELDS}
    out = {k: v.astype(np.float32 if k in ("value", "prior") else np.int64) for k, v in out.items()}
    out["used"] = used
    return out


def _same(got, want, what):
    assert got["used"] == want["used"], (what, got["used"], want["used"])
    for k in FIELDS:
        g, w = got[k], want[k]
        bad = np.flatnonzero(g.view(np.int32) != w.view(np.int32)) if g.dtype == np.float32 else np.flatnonzero(g != w)
        assert bad.size == 0, (what, k, bad[:8].tolist(), g[bad[:4]].tolist(), w[bad[:4]].tolist())


def _against_reference(e, version, dense, player, rows, rounds, max_nodes, c_puct=1.25, fpu=0.0, dtype=torch.float32,
                       net_of=None, after_round=None, log=None):
    """grow trees from the imported states round by round, each round's leaves and the final trees against the
    reference.  The network is net_of(b, leaf state, player, n_logits) -> (float32 logits, value), by default
    _guided_ref.net of the exported leaf state; the logits reach the device in `dtype` and the reference as the device
    reads them (rounded to dtype).  after_round(r, tree, refs) runs after each round's backups; log (a list) receives
    each round's (node, kind) arrays."""
    orc = logic(version)
    B = len(player)
    st = e.import_ref_state(torch.as_tensor(dense, device="cuda"),
                            torch.as_tensor(np.asarray(player, np.int8), device="cuda"))
    tree = e.guided_tree(st, max_nodes)
    refs = [GuidedTree(orc, dense[b], int(player[b]), max_nodes) for b in range(B)]
    n = e.layout.spatial_actions
    kinds = np.zeros(3, np.int64)
    if net_of is None:
        net_of = lambda b, s, p, n_logits: net(s, p, n_logits)  # noqa: E731
    for r in range(rounds):
        leaves = e.guided_select(st, tree, c_puct=c_puct, fpu=fpu)
        ld, lp = (x.cpu().numpy() for x in e.export_ref_state(leaves.states))
        node, kind = leaves.node.cpu().numpy(), leaves.kind.cpu().numpy()
        nets = [net_of(b, ld[b], int(lp[b]), n) for b in range(B)]
        logits = torch.as_tensor(np.stack([x for x, _ in nets])).to("cuda", dtype).view(B, *e.spatial_action_size)
        seen = logits.float().view(B, n).cpu().numpy()
        values = torch.as_tensor(np.array([v for _, v in nets], np.float32), device="cuda")
        e.guided_backup(tree, leaves, logits, values)
        prior = tree.prior.cpu().numpy()
        for b in range(B):
            v, s, p, k = refs[b].select(c_puct, fpu)
            what = (version, rows[b], r)
            assert (int(node[b]), int(kind[b])) == (v, k), (what, int(node[b]), int(kind[b]), v, k)
            assert np.array_equal(ld[b], s) and int(lp[b]) == p, what
            refs[b].backup(v, s, p, k, seen[b], nets[b][1], prior[b])
            kinds[k] += 1
        if log is not None:
            log.append((node, kind))
        if after_round is not None:
            after_round(r, tree, refs)
    for b in range(B):
        want = refs[b].arrays()
        _same(_host(tree, b), want, (version, rows[b]))
        check_invariants(want, rounds, max_nodes)
    return st, tree, kinds


@pytest.mark.parametrize("version", VERSIONS)
def test_trees_and_leaves_equal_the_reference(version):
    """24 rounds on recorded states (both players to move): c_puct 1.25 / fpu 0 with float32 logits, c_puct 0.5 /
    fpu -1 with bfloat16, c_puct 1.25 / fpu -1 with float16"""
    e = _engine(version)
    dense, player, rows = _recorded(version)
    _against_reference(e, version, dense, player, rows, 24, 2000)
    h = len(rows) // 2
    pick = [0, 1, h, h + 1, len(rows) - 1]
    sub = (dense[pick], player[pick], [rows[i] for i in pick])
    _against_reference(e, version, *sub, 20, 2000, c_puct=0.5, fpu=-1.0, dtype=torch.bfloat16)
    _against_reference(e, version, *sub, 20, 2000, c_puct=1.25, fpu=-1.0, dtype=torch.float16)


@pytest.mark.parametrize("version,row", [("barrage", 237), ("micro", 36), ("tiny", 181)])
def test_stuck_and_finished_roots(version, row):
    """a root whose player to move is stuck and finished roots stay used = 1 and back up their outcome every round"""
    e = _engine(version)
    t = traj(version)
    over = [i for i in range(t["states"].shape[0]) if t["states"][i][5][0, 1]][:2]
    dense = t["states"][[row] + over].astype(np.int64)
    player = np.array([-int(t["players"][row])] + [int(t["players"][i]) for i in over], np.int64)
    _, tree, kinds = _against_reference(e, version, dense, player, [row] + over, 12, 50)
    assert kinds[LEAF_STUCK] == 12 and kinds[LEAF_OVER] == 12 * len(over) and kinds[LEAF_EVAL] == 0
    assert bool((tree.used == 1).all()) and bool((tree.visits[:, 0] == 12).all())
    assert float(tree.value[0, 0]) == 12.0 * -int(player[0])  # the stuck player loses every round


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_pool_exhaustion(version):
    """pools of 1, 2, the first root's children plus one, and 70 nodes: expansions stop, values still back up"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 3)
    n_root = len(action_list(logic(version), dense[0], player[0]))
    for nodes in (1, 2, n_root + 1, 70):
        _, tree, _ = _against_reference(e, version, dense, player, rows, 16, nodes)
        assert bool((tree.used <= nodes).all()) and bool((tree.visits[:, 0] == 16).all())


def _device_net(e, leaves):
    """a deterministic evaluator on the device: logits (multiples of 1/8, some -inf) and values (multiples of 1/16)
    from the leaves' state keys"""
    B, n = leaves.node.shape[0], e.layout.spatial_actions
    h = (e.state_keys(leaves.states) >> 20) & 0xFFFF
    idx = torch.arange(n, device="cuda")
    x = ((h[:, None] * 31 + idx[None, :] * 7) * 2654435761) >> 13
    logits = ((x % 9) - 4).to(torch.float32) / 8
    logits = torch.where((h[:, None] * 13 + idx[None, :]) % 5 == 0, float("-inf"), logits)
    values = (((h * 40503) >> 4) % 33 - 16).to(torch.float32) / 16
    return logits.view(B, *e.spatial_action_size).contiguous(), values


def _rounds(e, st, tree, rounds, c_puct=1.25, fpu=0.0, record=None):
    """`rounds` rounds with the device evaluator; record (a dict row -> list) receives each round's logits and value
    of those rows"""
    for _ in range(rounds):
        leaves = e.guided_select(st, tree, c_puct=c_puct, fpu=fpu)
        logits, values = _device_net(e, leaves)
        if record is not None:
            for b, acc in record.items():
                acc.append((logits[b].reshape(-1).cpu().numpy(), np.float32(values[b].item())))
        e.guided_backup(tree, leaves, logits, values)
    return tree


def _tree_rows(tree):
    """the fields of every tree with the unused columns zeroed (they hold anything)"""
    M = tree.visits.shape[1]
    live = torch.arange(M, device="cuda")[None, :] < tree.used.long()[:, None]
    out = {"used": tree.used}
    for k in TREE[:-1]:
        t = getattr(tree, k)
        out[k] = torch.where(live, t, torch.zeros((), dtype=t.dtype, device="cuda"))
    return out


@pytest.mark.parametrize("version", ["barrage", "standard", "standard2", "micro", "fives"])
def test_root_children_and_read_only_parts(version):
    """on de-phased self-play games: the root's children equal expand_moves(state).actions; the roots are never
    written; a select leaves the tree untouched and a second select returns the same leaves"""
    e = _engine(version)
    st = _selfplay(e, 512, 60, seed=4)
    before = st.clone()
    tree = _rounds(e, st, e.guided_tree(st, 600), 6)
    for n in STATE:
        assert torch.equal(getattr(st, n), getattr(before, n)), n
    ex = e.expand_moves(st)
    off = ex.offsets.cpu()
    for b in range(st.num_envs):
        f, n = int(tree.first_child[b, 0]), int(tree.n_children[b, 0])
        got = tree.action[b, f:f + n] if f >= 0 else tree.action[b, :0]
        assert torch.equal(got, ex.actions[off[b]:off[b + 1]]), (version, b)
    bits = lambda t: t.view(torch.int32) if t.dtype == torch.float32 else t  # noqa: E731  (unused columns may hold NaN)
    snap = {k: bits(getattr(tree, k)).clone() for k in TREE}
    a = e.guided_select(st, tree, c_puct=0.8, fpu=-0.25)
    b = e.guided_select(st, tree, c_puct=0.8, fpu=-0.25)
    for k in TREE:
        assert torch.equal(bits(getattr(tree, k)), snap[k]), k
    for n in STATE:
        assert torch.equal(getattr(st, n), getattr(before, n)), n
        assert torch.equal(getattr(a.states, n), getattr(b.states, n)), n
    assert torch.equal(a.node, b.node) and torch.equal(a.kind, b.kind)


def test_deterministic_and_independent_of_the_batch_split():
    """two runs give identical trees; rows [lo, hi) grown alone equal those rows"""
    e = _engine("barrage")
    st = _selfplay(e, 300, 80, seed=2)
    x = _tree_rows(_rounds(e, st, e.guided_tree(st, 900), 24))
    y = _tree_rows(_rounds(e, st, e.guided_tree(st, 900), 24))
    for k in TREE:
        assert torch.equal(x[k], y[k]), k
    lo, hi = 70, 211
    part = st.select(lo, hi)
    part = type(part)(*(getattr(part, n).contiguous() for n in STATE))
    z = _tree_rows(_rounds(e, part, e.guided_tree(part, 900), 24))
    for k in TREE:
        assert torch.equal(z[k], x[k][lo:hi]), k


def test_a_round_does_not_synchronise_the_host():
    e = _engine("barrage")
    st = _selfplay(e, 256, 40, seed=5)
    tree = e.guided_tree(st, 500)
    leaves = e.guided_select(st, tree)
    logits, values = _device_net(e, leaves)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        tree = e.guided_tree(st, 500)
        leaves = e.guided_select(st, tree)
        e.guided_backup(tree, leaves, logits, values)
        leaves = e.guided_select(st, tree, c_puct=0.5, fpu=-1.0)
        e.guided_backup(tree, leaves, logits.to(torch.bfloat16), values)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert bool((tree.visits[:, 0] == 2).all())


def _device_invariants(tree, rounds):
    """the contract's consequences on every tree, with torch ops"""
    B, M = tree.visits.shape
    used = tree.used.long()
    cols = torch.arange(M, device="cuda")[None, :]
    live = cols < used[:, None]
    assert bool((used >= 1).all()) and bool((used <= M).all())
    assert bool((tree.visits[:, 0] == rounds).all()) and bool((tree.parent[:, 0] == -1).all())
    N = torch.where(live, tree.visits, 0).long()
    par = tree.parent.long()
    child = live & (cols > 0)
    assert bool(((par >= 0) & (par < cols))[child].all())
    slot = torch.where(child, par, M)
    kid_sum = torch.zeros(B, M + 1, dtype=torch.long, device="cuda").scatter_add_(1, slot, N)[:, :M]
    kid_n = torch.zeros(B, M + 1, dtype=torch.long, device="cuda").scatter_add_(1, slot, child.long())[:, :M]
    p_sum = torch.zeros(B, M + 1, dtype=torch.float64, device="cuda").scatter_add_(
        1, slot, torch.where(child, tree.prior.double(), 0.0))[:, :M]
    fc, nc = tree.first_child.long(), tree.n_children.long()
    expanded = live & (fc >= 0)
    assert bool((N == kid_sum + 1)[expanded].all())
    assert bool((nc == kid_n)[live].all())
    assert bool(((fc + nc <= used[:, None]) & (fc > cols))[expanded].all())
    assert bool(((p_sum - 1).abs() <= nc.double() * 2.0 ** -23)[expanded].all())
    W = torch.where(live, tree.value, 0.0)
    assert bool((W.abs() <= N.float())[live].all())  # every value backed up lies in [-1, 1]


def test_full_size_barrage():
    """65 536 de-phased Barrage trees x 64 rounds with the device evaluator: the invariants on every tree and the
    reference on sampled rows, given the logits and values the device evaluator gave those rows"""
    e = _engine("barrage")
    B, R, M = 65536, 64, 2048
    st = _selfplay(e, B, 200, seed=8)
    rows = (0, 1, 777, 40000, 65535)
    record = {b: [] for b in rows}
    tree = _rounds(e, st, e.guided_tree(st, M), R, record=record)
    _device_invariants(tree, R)
    dense, player = (x.cpu().numpy() for x in e.export_ref_state(st))
    orc = logic("barrage")
    prior = tree.prior[list(rows)].cpu().numpy()
    for i, b in enumerate(rows):
        ref = GuidedTree(orc, dense[b], int(player[b]), M)
        for logits, value in record[b]:
            v, s, p, k = ref.select(1.25, 0.0)
            ref.backup(v, s, p, k, logits, value, prior[i])
        _same(_host(tree, b), ref.arrays(), b)


def test_batched_env_forwards_its_games():
    from stratego_env_b200.batched_env import BatchedStrategoEnv
    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=64, device="cuda:0", seed=3, env_base=1000)
    env.reset()
    e = env.engine
    tree, want = env.guided_tree(300), e.guided_tree(env.state, 300)
    for _ in range(5):
        leaves, ref = env.guided_select(tree, c_puct=0.9), e.guided_select(env.state, want, c_puct=0.9)
        assert torch.equal(leaves.node, ref.node) and torch.equal(leaves.kind, ref.kind)
        for n in STATE:
            assert torch.equal(getattr(leaves.states, n), getattr(ref.states, n)), n
        logits, values = _device_net(e, leaves)
        e.guided_backup(tree, leaves, logits, values)
        e.guided_backup(want, ref, logits, values)
    x, y = _tree_rows(tree), _tree_rows(want)
    for k in TREE:
        assert torch.equal(x[k], y[k]), k
    visits, values = tree.root_stats()
    assert visits.dtype == torch.int32 and values.dtype == torch.float32 and int(visits.sum()) == 64 * 4
