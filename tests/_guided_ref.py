"""Reference of the guided tree search (sx_guided_select / sx_guided_backup), on the reference's dense state layout.

One tree per root, node 0 the root, fields as in include/stratego_b200.h, W and P float32.  select() descends from the
root by the numpy float32 PUCT score (one rounding per operation, ties to the lowest index) to the first node without
children or whose state is over; the step is the oracle's maenv:684-692 step (orc.apply_spatial_action).  backup()
expands an evaluable leaf without children into the _expand_ref.action_list moves when the pool has room, with priors
checked against the float64 softmax of the logits over the legal entries (within prior_bound) and then taken from the
device (the only transcendental result), and adds the value to N and W (float32) along the path.  softmax_f32 emulates
the kernel's float32 softmax, so that the bound can be checked without a device.  net() is a deterministic "network" of
the dense state for the tests: logits are small multiples of 1/8 with ties and some -inf entries, the value a multiple
of 1/16, so float32, bfloat16 and float16 hold them exactly."""
import numpy as np

from _expand_ref import action_list
from _keys_ref import state_keys_ref
from _playout_ref import INVALID, OVER, WINNER, data

LEAF_EVAL, LEAF_OVER, LEAF_STUCK = 0, 1, 2
FIELDS = ("visits", "value", "parent", "first_child", "n_children", "action", "prior")
f32 = np.float32


def net(dense, player, n_logits):
    """(logits float32 [n_logits], value float32) of a dense state: drawn from a generator seeded by the state key"""
    key = int(state_keys_ref(np.asarray(dense, np.int64)[None], [int(player)])[0])
    rng = np.random.default_rng(key)
    logits = (rng.integers(-4, 5, n_logits) / 8).astype(f32)
    style = key % 8
    if style == 0:
        logits[:] = -np.inf  # every entry -inf: uniform priors
    elif style < 4:
        logits[rng.random(n_logits) < 0.3] = -np.inf
    value = f32(rng.integers(-16, 17) / 16)
    return logits, value


LOGIT_CASES = ("sigma1", "sigma4", "sigma10", "sigma30", "dominant", "extremes", "all_inf")


def network_logits(rng, case, n, big):
    """float32 [n]: logits of n legal moves as a policy head gives them.  sigmaS: N(0, S); dominant: one logit near 5,
    the others more than 110 below it (their priors are exactly 0 in float32, also after rounding to bfloat16 / float16);
    extremes: +-big (the dtype's largest finite value) mixed with N(0, 3); all_inf: every entry -inf"""
    if case.startswith("sigma"):
        return (rng.standard_normal(n) * float(case[5:])).astype(f32)
    if case == "dominant":
        x = 5 + rng.standard_normal() - 112 - np.abs(rng.standard_normal(n)) * 8
        x[rng.integers(n)] = 5 + rng.standard_normal()
        return x.astype(f32)
    if case == "extremes":
        x = rng.standard_normal(n) * 3
        r = rng.random(n)
        x[r < 0.15], x[(r >= 0.15) & (r < 0.3)] = big, -big
        return x.astype(f32)
    assert case == "all_inf", case
    return np.full(n, -np.inf, f32)


def scores(W, N, P, n_parent, sigma, c_puct, fpu):
    """numpy float32 PUCT scores of children (W, N, P) of a node with n_parent visits, as the kernel rounds them"""
    W, P = np.asarray(W, f32), np.asarray(P, f32)
    N = np.asarray(N, np.int64)
    visited = N > 0
    q = np.where(visited, (f32(sigma) * W) / np.maximum(N, 1).astype(f32), f32(fpu)).astype(f32)
    u = ((f32(c_puct) * P) * np.sqrt(f32(n_parent))) / (1 + N).astype(f32)
    return (q + u).astype(f32)


def softmax64(x):
    """float64 softmax of the legal logits; 1/n each when all are -inf"""
    x = np.asarray(x, np.float64)
    if not np.any(x > -np.inf):
        return np.full(x.size, 1.0 / x.size)
    e = np.exp(x - x.max())
    return e / e.sum()


def prior_bound(x):
    """float64 [n]: how far each float32 prior of the legal logits x may lie from the float64 softmax w,
    (n + 8 + |x - max|) * 2^-24 * w + 2^-146.  fl(x - max) is off by up to 2^-24 |x - max| absolute, which exp turns into
    the same relative error; n + 8 covers the float32 sum, expf's 2 ulp and the division; 2^-146 covers priors that
    round into or below the subnormal range.  An entry at -inf (w = 0) counts |x - max| as 0."""
    x = np.asarray(x, np.float64)
    w = softmax64(x)
    y = np.abs(x - x.max()) if np.any(x > -np.inf) else np.zeros(x.size)
    y = np.where(np.isfinite(y), y, 0.0)
    return (x.size + 8 + y) * 2.0 ** -24 * w + 2.0 ** -146


def check_priors(got, x):
    """device priors of one child block against the float64 softmax: each within prior_bound(x), the block's sum 1
    within n * 2^-23"""
    got = np.asarray(got, f32)
    want = softmax64(x)
    n = want.size
    err = np.abs(got.astype(np.float64) - want)
    assert np.all(err <= prior_bound(x)), (got.tolist(), want.tolist())
    assert abs(float(got.astype(np.float64).sum()) - 1.0) <= n * 2.0 ** -23, got.tolist()


def softmax_f32(x, exp_ulps=None):
    """the kernel's softmax of the legal logits x in numpy float32: fl(x - max), exp correctly rounded to float32 (then
    scaled by 1 + exp_ulps * 2^-23 if given, to stand for expf's error), a float32 sum in ascending order and a float32
    division; 1/n each when every entry is -inf"""
    x = np.asarray(x, f32)
    if not np.any(x > -np.inf):
        return np.full(x.size, f32(1) / f32(x.size), f32)
    with np.errstate(over="ignore"):
        y = x - x.max()  # float32 -FLT_MAX - FLT_MAX overflows to -inf, as __fsub_rn does
        e = np.exp(y.astype(np.float64)).astype(f32)
    if exp_ulps is not None:
        e = (e * (1 + np.asarray(exp_ulps, np.float64) * 2.0 ** -23)).astype(f32)
    s = np.cumsum(e, dtype=f32)[-1]  # add.accumulate is sequential: one float32 rounding per term
    return e / s


class GuidedTree:
    """one guided tree, grown by select() / backup() rounds as the device grows it"""

    def __init__(self, orc, root, player, max_nodes):
        self.orc, self.max_nodes = orc, int(max_nodes)
        self.t = dict(visits=[0], value=[f32(0)], parent=[-1], first_child=[-1], n_children=[0], action=[-1],
                      prior=[f32(1)])
        self.states = {0: (np.ascontiguousarray(root, dtype=np.int64), int(player))}  # node -> (dense, player to move)

    @property
    def used(self):
        return len(self.t["visits"])

    def select(self, c_puct, fpu):
        """(leaf node, dense state, player to move, kind)"""
        t = self.t
        v = 0
        s, p = self.states[0]
        while not data(s, OVER) and t["first_child"][v] >= 0:
            f, n = t["first_child"][v], t["n_children"][v]
            sc = scores(t["value"][f:f + n], t["visits"][f:f + n], t["prior"][f:f + n], t["visits"][v],
                        1 if p == 1 else -1, c_puct, fpu)
            c = f + int(np.argmax(sc))  # the first maximum: ties to the lowest index
            if c not in self.states:
                self.states[c] = self.orc.apply_spatial_action(s, p, t["action"][c])
            s, p = self.states[c]
            v = c
        if data(s, OVER):
            kind = LEAF_OVER
        else:
            kind = LEAF_EVAL if action_list(self.orc, s, p).size else LEAF_STUCK
        return v, s, p, kind

    def backup(self, v, s, p, kind, logits, value, device_prior):
        """expand and back up leaf v (state s, player p) with the network's logits (float32, flat) and value; the
        children's priors are checked against the float64 softmax and taken from device_prior (the device tree's P; None:
        the float64 softmax rounded to float32)"""
        t = self.t
        sigma = 1 if p == 1 else -1
        if kind == LEAF_EVAL and t["first_child"][v] < 0:
            acts = action_list(self.orc, s, p)
            n = acts.size
            if n and self.used + n <= self.max_nodes:
                f = self.used
                x = np.asarray(logits, f32)[acts]
                if device_prior is None:  # no device: the float64 softmax rounded to float32
                    got = softmax64(x).astype(f32)
                else:
                    got = np.asarray(device_prior[f:f + n], f32)
                    check_priors(got, x)
                t["first_child"][v], t["n_children"][v] = f, n
                for a, pr in zip(acts, got):
                    for k, val in zip(FIELDS, (0, f32(0), v, -1, 0, int(a), f32(pr))):
                        t[k].append(val)
        if kind == LEAF_EVAL:
            z = f32(sigma) * f32(value)
        elif kind == LEAF_OVER:
            z = f32(0 if data(s, INVALID) else data(s, WINNER))
        else:
            z = f32(-sigma)
        x = v
        while x >= 0:
            t["visits"][x] += 1
            t["value"][x] = f32(t["value"][x] + z)
            x = t["parent"][x]

    def set_prior(self, first, values):
        """the caller's rewrite of P of nodes first, first + 1, ... (float32), as on the device between calls"""
        for k, val in enumerate(np.asarray(values, f32)):
            self.t["prior"][first + k] = f32(val)

    def arrays(self):
        """dict of arrays [used] per field of FIELDS (W and P float32, the rest int64), and "used" """
        out = {k: np.array(self.t[k], dtype=f32 if k in ("value", "prior") else np.int64) for k in FIELDS}
        out["used"] = self.used
        return out


def check_invariants(tree, rounds, max_nodes):
    """the contract's consequences on one tree (arrays()): root N = rounds, N = 1 + the children's N on every expanded
    node, links and pool use, children in ascending action order"""
    used = int(tree["used"])
    N, parent, fc, nc, act = (np.asarray(tree[k])[:used] for k in ("visits", "parent", "first_child", "n_children",
                                                                     "action"))
    assert 1 <= used <= max_nodes
    assert N[0] == rounds and parent[0] == -1 and act[0] == -1
    for j in range(used):
        if fc[j] < 0:
            assert nc[j] == 0
            continue
        kids = np.arange(fc[j], fc[j] + nc[j])
        assert nc[j] > 0 and kids[-1] < used
        assert np.all(parent[kids] == j)
        assert np.all(np.diff(act[kids]) > 0)
        assert N[j] == 1 + N[kids].sum(), j
    assert np.all(parent[1:] < np.arange(1, used))
