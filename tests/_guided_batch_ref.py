"""Reference of guided tree search with L leaves per tree and round under a virtual loss (sx_guided_select_many /
sx_guided_backup_many), built on _guided_ref.GuidedTree, whose functions it leaves as they are.

select_many() chooses the L leaves of a round in order, each a full descent from the root; before leaf j, every node on
the paths of leaves 0 .. j-1 carries V = the number of those paths through it, and scores_vl gives the virtual-visit
score in numpy float32 (one rounding per operation).  backup_many() takes the leaves in order with GuidedTree.backup,
so an EVAL leaf is expanded only if its node has no children at that point (a node reached by several leaves of a round
is expanded once, by the first of them) and every leaf backs up its own value.  `ends` counts the selections that
ended at each node, for check_invariants_many: N = e + the sum of the children's N on every node."""
import numpy as np

from _expand_ref import action_list
from _guided_ref import LEAF_EVAL, LEAF_OVER, LEAF_STUCK, GuidedTree
from _playout_ref import OVER, data

f32 = np.float32


def scores_vl(W, N, V, P, n_parent, v_parent, sigma, c_puct, fpu, vl):
    """numpy float32 scores of children (W, N, V, P) of a node with n_parent visits and v_parent pending visits:
    n = N + V, q = n > 0 ? (sigma * W - vl * float(V)) / float(n) : fpu, u = ((c_puct * P) * sqrt(N_v + V_v)) / (1 + n)"""
    W, P = np.asarray(W, f32), np.asarray(P, f32)
    N, V = np.asarray(N, np.int64), np.asarray(V, np.int64)
    n = N + V
    with np.errstate(over="ignore", invalid="ignore"):
        q = np.where(n > 0, (f32(sigma) * W - f32(vl) * V.astype(f32)) / np.maximum(n, 1).astype(f32), f32(fpu))
        u = ((f32(c_puct) * P) * np.sqrt(f32(int(n_parent) + int(v_parent)))) / (1 + n).astype(f32)
        return (q.astype(f32) + u).astype(f32)


class BatchTree(GuidedTree):
    """one guided tree grown by rounds of L leaves, as the device grows it"""

    def __init__(self, orc, root, player, max_nodes):
        super().__init__(orc, root, player, max_nodes)
        self.ends = {}  # node -> selections that ended there

    def select_many(self, L, c_puct, fpu, vl):
        """the round's L leaves in order: [(leaf node, dense state, player to move, kind)]"""
        t = self.t
        V = np.zeros(self.used, np.int64)
        out = []
        for _ in range(L):
            v = 0
            s, p = self.states[0]
            while not data(s, OVER) and t["first_child"][v] >= 0:
                f, n = t["first_child"][v], t["n_children"][v]
                sc = scores_vl(t["value"][f:f + n], t["visits"][f:f + n], V[f:f + n], t["prior"][f:f + n],
                               t["visits"][v], V[v], 1 if p == 1 else -1, c_puct, fpu, vl)
                c = f + int(np.argmax(sc))  # the first maximum: ties to the lowest index
                if c not in self.states:
                    self.states[c] = self.orc.apply_spatial_action(s, p, t["action"][c])
                s, p = self.states[c]
                v = c
            if data(s, OVER):
                kind = LEAF_OVER
            else:
                kind = LEAF_EVAL if action_list(self.orc, s, p).size else LEAF_STUCK
            out.append((v, s, p, kind))
            x = v
            while x >= 0:
                V[x] += 1
                x = t["parent"][x]
        return out

    def backup_many(self, leaves, logits, values, device_prior):
        """back up the round's leaves in order; logits[j] (float32, flat) and values[j] belong to leaves[j]"""
        for (v, s, p, kind), x, z in zip(leaves, logits, values):
            self.backup(v, s, p, kind, x, z, device_prior)
            self.ends[v] = self.ends.get(v, 0) + 1


def check_invariants_many(tree, ends, max_nodes):
    """the contract's consequences on one tree (arrays()) after rounds whose leaves ended at `ends` (node -> count):
    root N = the number of leaves, N = e + the children's N on every node, links and pool use, children in ascending
    action order"""
    used = int(tree["used"])
    N, parent, fc, nc, act = (np.asarray(tree[k])[:used] for k in ("visits", "parent", "first_child", "n_children",
                                                                     "action"))
    e = np.zeros(used, np.int64)
    for v, k in ends.items():
        e[v] += k
    assert 1 <= used <= max_nodes
    assert N[0] == e.sum() and parent[0] == -1 and act[0] == -1
    kid_sum = np.zeros(used, np.int64)
    np.add.at(kid_sum, parent[1:], N[1:])
    assert np.array_equal(N, e + kid_sum), np.flatnonzero(N != e + kid_sum)[:8]
    for j in range(used):
        if fc[j] < 0:
            assert nc[j] == 0
            continue
        kids = np.arange(fc[j], fc[j] + nc[j])
        assert nc[j] > 0 and kids[-1] < used
        assert np.all(parent[kids] == j)
        assert np.all(np.diff(act[kids]) > 0)
    assert np.all(parent[1:] < np.arange(1, used))
