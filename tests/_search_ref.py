"""Reference of the device tree search (sx_search), on the reference's dense state layout.

One tree per root, node 0 the root, fields as in include/stratego_b200.h.  Iteration i descends from the root: at a
node without children the action list of _expand_ref.action_list (ascending flat spatial index) becomes its children
when the pool has room; the child is the first one with N = 0, else the argmax of the numpy float32 PUCT score (ties to
the lowest index); the step is the oracle's maenv:684-692 step (orc.apply_spatial_action).  The state reached is scored
by its outcome or by a playout with the rules of _playout_ref and the search's draw: Philox4x32-10 (_sampler_ref),
counter (gid lo, gid hi, RNG_SEARCH ^ i, turn & 0xffff), first word, uniform_valid_ref over the mask of the player to
move.  The score z is added to N and W of every node on the path."""
import numpy as np

from _expand_ref import action_list
from _playout_ref import INVALID, OVER, TURN, WINNER, data
from _sampler_ref import _key, philox4x32_10, uniform_valid_ref

RNG_SEARCH = 0x54524545
FIELDS = ("visits", "value", "parent", "first_child", "n_children", "action")


def search_word(gid, it, turn, seed):
    """first Philox word of the search's playout draw"""
    k0, k1 = _key(seed)
    gid = int(gid) & (2 ** 64 - 1)
    return philox4x32_10(np.array([gid & 0xFFFFFFFF]), np.array([gid >> 32]), np.array([(RNG_SEARCH ^ int(it)) & 0xFFFFFFFF]),
                         np.array([int(turn) & 0xFFFF]), k0, k1)[0]


def outcome(state):
    """player +1's reward of a finished state: the winner, 0 for a turn-limit ending"""
    return 0 if data(state, INVALID) else data(state, WINNER)


def search_playout(orc, state, player, gid, it, seed, max_plies):
    """z of a playout of at most max_plies plies (0 if cut off), and the plies played"""
    plies = 0
    while plies < max_plies and not data(state, OVER):
        mask, _, _ = orc.current_obs(state, player, obs_mode=0)
        A = mask.shape[-1]
        a = int(uniform_valid_ref(mask.reshape(1, -1), search_word(gid, it, data(state, TURN), seed))[0])
        if a == A - 1:  # the noop entry is the whole mask: the player to move is stuck and loses
            state, player = orc.base_env.get_next_state(state, player, orc.base_env.action_size - 1)
        else:
            state, player = orc.apply_spatial_action(state, player, a)
        plies += 1
    return (outcome(state) if data(state, OVER) else 0), plies


def score(W, N, n_parent, sigma, c_explore):
    """numpy float32 PUCT scores of children with counts N, W (all N > 0), as the kernel rounds them"""
    f = np.float32
    q = (sigma * np.asarray(W, np.int64)).astype(f) / np.asarray(N).astype(f)
    u = (f(c_explore) * np.sqrt(f(n_parent))) / (1 + np.asarray(N)).astype(f)
    return (q + u).astype(f)


def search_ref(orc, root, player, gid, seed, iterations, max_nodes, max_plies, c_explore, stats=None):
    """dict of int64 arrays [used] per field of FIELDS, and "used"; stats (a dict) receives the playout plies"""
    root = np.ascontiguousarray(root, dtype=np.int64)
    t = {k: [0] for k in ("visits", "value")}
    t.update(parent=[-1], first_child=[-1], n_children=[0], action=[-1])
    states = {0: (root, int(player))}  # node -> (dense state, player to move), cached
    plies_total = 0
    for it in range(iterations):
        v = 0
        s, p = states[0]
        path = [0]
        while not data(s, OVER):
            if t["first_child"][v] < 0:
                acts = action_list(orc, s, p)
                n = len(acts)
                if n == 0 or len(t["visits"]) + n > max_nodes:
                    break
                t["first_child"][v], t["n_children"][v] = len(t["visits"]), n
                for a in acts:
                    for k, x in zip(FIELDS, (0, 0, v, -1, 0, int(a))):
                        t[k].append(x)
            f, n = t["first_child"][v], t["n_children"][v]
            N = np.array(t["visits"][f:f + n])
            zero = np.flatnonzero(N == 0)
            if zero.size:
                j = int(zero[0])
            else:
                sc = score(t["value"][f:f + n], N, t["visits"][v], 1 if p == 1 else -1, c_explore)
                j = int(np.argmax(sc))
            c = f + j
            if c not in states:
                states[c] = orc.apply_spatial_action(s, p, t["action"][c])
            s, p = states[c]
            v = c
            path.append(c)
            if zero.size:
                break
        if data(s, OVER):
            z = outcome(s)
        else:
            z, n_plies = search_playout(orc, s, p, gid, it, seed, max_plies)
            plies_total += n_plies
        for x in path:
            t["visits"][x] += 1
            t["value"][x] += z
    if stats is not None:
        stats["plies"] = plies_total
    out = {k: np.array(t[k], dtype=np.int64) for k in FIELDS}
    out["used"] = len(t["visits"])
    return out


def check_invariants(tree, iterations, max_nodes):
    """the consequences of the contract that hold for any tree: root counts, N sums, parent / child links, pool use"""
    used = int(tree["used"])
    N, parent, fc, nc, act = (np.asarray(tree[k])[:used] for k in ("visits", "parent", "first_child", "n_children",
                                                                     "action"))
    W = np.asarray(tree["value"])[:used]
    assert 1 <= used <= max_nodes
    assert N[0] == iterations and parent[0] == -1 and act[0] == -1
    assert np.all(np.abs(W) <= N)
    if iterations == 0:
        assert used == 1
    for j in range(used):
        if fc[j] < 0:
            assert nc[j] == 0
            continue
        kids = np.arange(fc[j], fc[j] + nc[j])
        assert nc[j] > 0 and kids[-1] < used
        assert np.all(parent[kids] == j)
        assert np.all(np.diff(act[kids]) > 0)  # ascending flat index
        assert N[j] == N[kids].sum() + (0 if j == 0 else 1), j
    assert np.all(parent[1:] < np.arange(1, used))
    # every non-root node is one of its parent's children
    for j in range(1, used):
        assert fc[parent[j]] <= j < fc[parent[j]] + nc[parent[j]]
