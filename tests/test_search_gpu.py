"""sx_search on the device: the whole tree (six node fields and used) against the reference of tests/_search_ref.py on
recorded states of every variant; pool exhaustion, finished, stuck, ply-capped and empty searches; the root's children
against expand_moves; the state left alone; determinism and the batch split; root_stats; a full-size batch."""
import numpy as np
import pytest
import torch

from _expand_ref import logic
from _golden import VERSIONS, traj
from _search_ref import FIELDS, check_invariants, search_ref
from test_expand_moves_gpu import _engine, _import, _selfplay

pytestmark = pytest.mark.gpu

SEED = 0xABCD_0000_1234_5678
BASE = 5 << 32
STATE = ("board", "aux", "captured")


def _sub(st, rows):
    from stratego_env_b200.engine import DeviceState
    idx = torch.as_tensor(rows, dtype=torch.long, device="cuda")
    return DeviceState(*(getattr(st, n).index_select(0, idx).contiguous() for n in STATE))


def _host(tree, b):
    """tree b as the reference returns it: the used columns of every field"""
    used = int(tree.used[b])
    out = {k: getattr(tree, k)[b, :used].cpu().numpy().astype(np.int64) for k in FIELDS}
    out["used"] = used
    return out


def _same(got, want, what):
    assert got["used"] == want["used"], (what, got["used"], want["used"])
    for k in FIELDS:
        bad = np.flatnonzero(got[k] != want[k])
        assert bad.size == 0, (what, k, bad[:8].tolist(), got[k][bad[:4]].tolist(), want[k][bad[:4]].tolist())


def _against_reference(e, version, dense, player, rows, iterations, max_nodes, max_plies, c_explore=1.0, seed=SEED,
                       env_base=BASE):
    """search the imported states and compare every tree with the reference"""
    orc = logic(version)
    st = e.import_ref_state(torch.as_tensor(dense, device="cuda"),
                            torch.as_tensor(np.asarray(player, np.int8), device="cuda"))
    tree = e.search(st, iterations, max_nodes=max_nodes, max_plies=max_plies, c_explore=c_explore, seed=seed,
                    env_base=env_base)
    M = tree.visits.shape[1]
    cap = (1 << 31) - 1 if max_plies is None else max_plies
    for b in range(len(player)):
        want = search_ref(orc, dense[b], int(player[b]), env_base + b, seed, iterations, M, cap, c_explore)
        _same(_host(tree, b), want, (version, rows[b]))
        check_invariants(want, iterations, M)
    return st, tree


def _recorded(version, k=6):
    """k recorded states spread over the trajectory (a game start first), each with both players to move"""
    t = traj(version)
    n = t["states"].shape[0]
    rows = sorted({int(np.flatnonzero(t["game_start"])[0]), *np.linspace(0, n - 1, k).astype(int).tolist()})
    dense = t["states"][rows].astype(np.int64)
    player = t["players"][rows].astype(np.int64)
    return (np.concatenate([dense, dense]), np.concatenate([player, -player]),
            rows + ["%d flipped" % r for r in rows])


@pytest.mark.parametrize("version", VERSIONS)
def test_trees_equal_the_reference(version):
    """64 iterations, playouts of at most 24 plies, the default pool, c_explore 1.0 and 0.35"""
    e = _engine(version)
    dense, player, rows = _recorded(version)
    _against_reference(e, version, dense, player, rows, 64, None, 24)
    _against_reference(e, version, dense[:4], player[:4], rows[:4], 40, None, 16, c_explore=0.35, seed=3, env_base=7)


def test_micro_to_the_end():
    """Micro, playouts to the end of the game"""
    e = _engine("micro")
    dense, player, rows = _recorded("micro", 10)
    _against_reference(e, "micro", dense, player, rows, 96, None, None)


@pytest.mark.parametrize("version", ["barrage", "standard", "micro"])
def test_pool_exhaustion(version):
    """pools of 1, 2, the root's children plus one, and 70 nodes: expansions stop when the children do not fit"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 3)
    for nodes in (1, 2, 41, 70):
        _, tree = _against_reference(e, version, dense, player, rows, 48, nodes, 12)
        assert bool((tree.used <= nodes).all())
    _, tree = _against_reference(e, version, dense[:2], player[:2], rows[:2], 30, 1, 20)
    assert bool((tree.used == 1).all()) and bool((tree.visits[:, 0] == 30).all())


@pytest.mark.parametrize("version,row", [("barrage", 237), ("micro", 36), ("tiny", 181)])
def test_stuck_and_finished_roots(version, row):
    """an imported root whose player to move is stuck is never expanded and loses every playout; a finished root is
    never expanded and scores its outcome every iteration"""
    e = _engine(version)
    t = traj(version)
    over = [i for i in range(t["states"].shape[0]) if t["states"][i][5][0, 1]][:2]
    dense = t["states"][[row] + over].astype(np.int64)
    player = np.array([-int(t["players"][row])] + [int(t["players"][i]) for i in over], np.int64)
    _, tree = _against_reference(e, version, dense, player, [row] + over, 20, None, 8)
    assert bool((tree.used == 1).all()) and bool((tree.visits[:, 0] == 20).all())
    assert int(tree.value[0, 0]) == 20 * -int(player[0])  # the stuck player loses by its noop every time


@pytest.mark.parametrize("version", ["barrage", "fives"])
def test_no_plies_and_no_iterations(version):
    """max_plies = 0 scores every unfinished leaf 0; iterations = 0 writes the root alone"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 4)
    _against_reference(e, version, dense, player, rows, 50, None, 0)
    _, tree = _against_reference(e, version, dense, player, rows, 0, 5, 10)
    assert bool((tree.used == 1).all()) and bool((tree.visits[:, 0] == 0).all())
    assert bool((tree.first_child[:, 0] == -1).all()) and bool((tree.action[:, 0] == -1).all())


def _root_children(tree, b):
    f, n = int(tree.first_child[b, 0]), int(tree.n_children[b, 0])
    return tree.action[b, f:f + n] if f >= 0 else tree.action[b, :0]


@pytest.mark.parametrize("version", ["barrage", "standard", "standard2", "micro", "fives"])
def test_root_children_are_the_expand_list_and_state_is_kept(version):
    """on de-phased self-play games: the root's child actions equal expand_moves(state).actions per game, and the
    state is byte for byte what it was"""
    e = _engine(version)
    st = _selfplay(e, 512, 60, seed=4)
    before = st.clone()
    tree = e.search(st, 16, max_plies=10, seed=9)
    for n in STATE:
        assert torch.equal(getattr(st, n), getattr(before, n)), n
    ex = e.expand_moves(st)
    off = ex.offsets.cpu()
    for b in range(st.num_envs):
        want = ex.actions[off[b]:off[b + 1]]
        assert torch.equal(_root_children(tree, b), want), (version, b)


def test_deterministic_and_independent_of_the_batch_split():
    """two calls give identical trees; rows [lo, hi) searched alone with env_base = lo equal those rows"""
    e = _engine("barrage")
    st = _selfplay(e, 300, 80, seed=2)
    kw = dict(max_nodes=900, max_plies=40, seed=SEED)
    a, b = e.search(st, 32, env_base=BASE, **kw), e.search(st, 32, env_base=BASE, **kw)
    used = a.used.long()
    cols = torch.arange(900, device="cuda")[None, :] < used[:, None]
    assert torch.equal(a.used, b.used)
    for k in FIELDS:
        assert torch.equal(torch.where(cols, getattr(a, k), 0), torch.where(cols, getattr(b, k), 0)), k
    lo, hi = 70, 211
    part = e.search(st.select(lo, hi), 32, env_base=BASE + lo, **kw)
    assert torch.equal(part.used, a.used[lo:hi])
    for k in FIELDS:
        assert torch.equal(torch.where(cols[lo:hi], getattr(part, k), 0), torch.where(cols[lo:hi], getattr(a, k)[lo:hi], 0)), k
    other = e.search(st, 32, env_base=BASE + 1, **kw)
    assert not torch.equal(torch.where(cols, other.value, 0), torch.where(cols, a.value, 0))


@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_root_stats_against_a_host_scatter(version):
    e = _engine(version)
    st = _selfplay(e, 200, 50, seed=6)
    tree = e.search(st, 40, max_plies=30, seed=1)
    visits, values = tree.root_stats()
    R, C, A = e.spatial_action_size
    assert visits.shape == values.shape == (200, R, C, A) and visits.dtype == values.dtype == torch.int32
    aux = st.aux.cpu().numpy().view(np.uint16)
    mask = e.valid_mask(st).cpu().numpy().reshape(200, -1)
    mask[:, A - 1::A] = 0
    for b in range(200):
        h = _host(tree, b)
        sign = 1 if ((aux[b, 2] >> 4) & 1) == 0 else -1
        wv, ww = np.zeros(R * C * A, np.int64), np.zeros(R * C * A, np.int64)
        kids = np.flatnonzero(h["parent"] == 0)
        wv[h["action"][kids]] = h["visits"][kids]
        ww[h["action"][kids]] = sign * h["value"][kids]
        assert np.array_equal(visits[b].reshape(-1).cpu().numpy(), wv), b
        assert np.array_equal(values[b].reshape(-1).cpu().numpy(), ww), b
        if kids.size:
            assert np.array_equal(np.flatnonzero(wv.astype(bool) | (mask[b] != 0)), np.flatnonzero(mask[b])), b
            assert int(wv.sum()) == 40


def test_batched_env_forwards_state_and_env_base():
    from stratego_env_b200.batched_env import BatchedStrategoEnv
    env = BatchedStrategoEnv({"version": "barrage"}, num_envs=64, device="cuda:0", seed=3, env_base=1000)
    env.reset()
    tree = env.search(24, seed=5, max_plies=20)
    want = env.engine.search(env.state, 24, max_plies=20, seed=5, env_base=1000)
    assert torch.equal(tree.used, want.used) and torch.equal(tree.visits[:, 0], want.visits[:, 0])
    cols = torch.arange(tree.visits.shape[1], device="cuda")[None, :] < tree.used.long()[:, None]
    for k in FIELDS:
        assert torch.equal(torch.where(cols, getattr(tree, k), 0), torch.where(cols, getattr(want, k), 0)), k


def _device_invariants(tree, iterations):
    """the contract's consequences on every tree, with torch ops"""
    B, M = tree.visits.shape
    used = tree.used.long()
    cols = torch.arange(M, device="cuda")[None, :]
    live = cols < used[:, None]
    assert bool((used >= 1).all()) and bool((used <= M).all())
    assert bool((tree.visits[:, 0] == iterations).all()) and bool((tree.parent[:, 0] == -1).all())
    N, W = torch.where(live, tree.visits, 0).long(), torch.where(live, tree.value, 0).long()
    assert bool((W.abs() <= N).all())
    par = tree.parent.long()
    child = live & (cols > 0)
    assert bool(((par >= 0) & (par < cols))[child].all())
    kid_sum = torch.zeros(B, M + 1, dtype=torch.long, device="cuda")
    kid_sum.scatter_add_(1, torch.where(child, par, M), N)
    kid_sum = kid_sum[:, :M]
    fc, nc = tree.first_child.long(), tree.n_children.long()
    expanded = live & (fc >= 0)
    want = kid_sum + (cols > 0).long()
    assert bool((N == want)[expanded].all())
    assert bool((nc == 0)[live & ~expanded].all()) and bool((kid_sum == 0)[live & ~expanded].all())
    assert bool(((fc + nc <= used[:, None]) & (fc > cols))[expanded].all())


def test_full_size_barrage():
    """4 096 de-phased Barrage trees x 128 iterations, playouts of at most 100 plies: the invariants on every tree and
    the reference on sampled rows"""
    e = _engine("barrage")
    B = 4096
    st = _selfplay(e, B, 200, seed=8)
    tree = e.search(st, 128, max_plies=100, seed=SEED, env_base=BASE)
    _device_invariants(tree, 128)
    dense, player = (x.cpu().numpy() for x in e.export_ref_state(st))
    orc = logic("barrage")
    for b in (0, 1, 777, 2048, 4095):
        want = search_ref(orc, dense[b], int(player[b]), BASE + b, SEED, 128, tree.visits.shape[1], 100, 1.0)
        _same(_host(tree, b), want, b)
