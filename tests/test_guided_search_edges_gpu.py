"""sx_guided_select / sx_guided_backup at the edges a network and a long search reach, against tests/_guided_ref.py:
priors from network-like logits (N(0, sigma) up to sigma 30, a dominant logit, +-finfo.max, a single move, every logit
-inf) in all three dtypes, with the illegal entries and the noop channel never read; float32 values whose sums round;
deep lines to the turn limit and to won games; the score's extremes and ties across lanes and 32-child passes;
priors the caller rewrites (Dirichlet noise); root_stats of a guided tree."""
import numpy as np
import pytest
import torch

from _expand_ref import action_list, logic
from _golden import traj
from _guided_ref import LEAF_OVER, LOGIT_CASES, net, network_logits, scores
from _keys_ref import state_keys_ref
from _playout_ref import INVALID, OVER, TURN, data
from test_expand_moves_gpu import _engine
from test_guided_search_gpu import _against_reference, _host
from test_search_gpu import _recorded

pytestmark = pytest.mark.gpu

f32 = np.float32
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
DTYPE_IDS = ["f32", "bf16", "f16"]
FLT_MAX = float(np.finfo(f32).max)


def _key(s, p):
    return int(state_keys_ref(np.asarray(s, np.int64)[None], [int(p)])[0])


def _scouts():
    """a Standard position, player +1 and player -1 to move, with 83 legal moves each: both sides have the eight
    scouts spread over the open files and the back rows, so lanes hold many moves and a child block spans three
    32-child passes"""
    from oracle.binding import OracleProceduralEnv
    env = OracleProceduralEnv(10, 10)
    lakes = np.zeros((10, 10), np.int64)
    for rc in [(4, 2), (5, 2), (4, 3), (5, 3), (4, 6), (5, 6), (4, 7), (5, 7)]:
        lakes[rc] = 1
    side = np.zeros((10, 10), np.int64)
    side[0, 0], side[0, 1], side[1, 0], side[0, 9] = 11, 12, 12, 10  # flag, two bombs, marshal
    for rc in [(1, 1), (2, 4), (3, 5), (1, 8), (2, 9), (3, 0), (0, 4), (0, 5)]:
        side[rc] = 2
    s = np.asarray(env.create_initial_state(lakes, side, side.copy(), 2000), np.int64)
    orc = logic("standard")
    for p in (1, -1):
        assert len(action_list(orc, s, p)) == 83, p
    return np.stack([s, s]), np.array([1, -1], np.int64)


# ---- priors from network-like logits --------------------------------------------------------------------------------
PRIOR_CASES = LOGIT_CASES + ("garbage", "clean")  # garbage / clean: sigma4 logits, illegal entries NaN / +inf or 0


def _prior_states(version):
    """(engine version, dense, player, labels): recorded states with both players to move, the 83-move Standard
    position, and recorded states whose player to move has a single legal move"""
    if version == "scouts":
        dense, player = _scouts()
        return "standard", dense, player, ["scouts +1", "scouts -1"]
    dense, player, rows = _recorded(version, 2)
    t = traj(version)
    orc = logic(version)
    single = [i for i in range(t["states"].shape[0]) if not data(t["states"][i], OVER)
              and len(action_list(orc, t["states"][i], t["players"][i])) == 1][:2]
    if single:
        dense = np.concatenate([dense, t["states"][single].astype(np.int64)])
        player = np.concatenate([player, t["players"][single].astype(np.int64)])
        rows = rows + ["%d single" % i for i in single]
    return version, dense, player, rows


@pytest.mark.parametrize("dtype", DTYPES, ids=DTYPE_IDS)
@pytest.mark.parametrize("version", ["barrage", "standard", "standard2", "micro", "scouts"])
def test_priors_from_network_like_logits(version, dtype):
    """every state under every case of PRIOR_CASES, 8 rounds: the trees and leaves against the reference (each prior
    within prior_bound of the float64 softmax of the dtype-rounded logits); then exact results: a dominant logit gives
    one prior 1 and the rest 0, every logit -inf gives 1/n each, a single move gets P = 1, and NaN / +inf in the
    illegal entries and the noop channel give the trees that 0 there gives"""
    engine_version, dense, player, rows = _prior_states(version)
    e = _engine(engine_version)
    orc = logic(engine_version)
    big = float(torch.finfo(dtype).max)
    C = len(PRIOR_CASES)
    case_of = [PRIOR_CASES[b % C] for b in range(len(player) * C)]

    def net_of(b, s, p, n_logits):
        case = case_of[b]
        base = "sigma4" if case in ("garbage", "clean") else case
        rng = np.random.default_rng([_key(s, p), LOGIT_CASES.index(base)])
        x = np.zeros(n_logits, f32)
        legal = action_list(orc, s, p)
        if legal.size:
            x[legal] = network_logits(rng, base, legal.size, big)
        if case == "garbage":
            off = np.ones(n_logits, bool)
            off[legal] = False
            x[off] = np.where(np.arange(n_logits)[off] % 2 == 0, np.nan, np.inf)
        return x, f32(rng.integers(-30, 31) * 0.1)

    rep = lambda a: np.repeat(a, C, axis=0)  # noqa: E731
    labels = [(rows[b // C], case_of[b]) for b in range(len(case_of))]
    _, tree, _ = _against_reference(e, engine_version, rep(dense), rep(player), labels, 8, 3000, dtype=dtype,
                                    net_of=net_of)
    hosts = [_host(tree, b) for b in range(len(case_of))]
    seen = set()
    for b, h in enumerate(hosts):
        for j in np.flatnonzero(h["first_child"] >= 0):
            f, n = h["first_child"][j], h["n_children"][j]
            P = h["prior"][f:f + n]
            if n == 1:
                assert P[0] == 1, labels[b]
                seen.add("single")
            if case_of[b] == "dominant":
                assert np.sort(P).tolist() == [0.0] * (n - 1) + [1.0], labels[b]
                seen.add("dominant")
            elif case_of[b] == "all_inf":
                assert np.all(P == f32(1) / f32(n)), labels[b]
                seen.add("all_inf")
    for b in range(len(case_of)):
        if case_of[b] == "garbage":
            want = hosts[b + 1]  # "clean" follows "garbage" in PRIOR_CASES
            assert case_of[b + 1] == "clean"
            for k in want:
                got = hosts[b][k]
                same = got == want[k] if k == "used" else np.array_equal(got.view(np.int32), want[k].view(np.int32)) \
                    if got.dtype == f32 else np.array_equal(got, want[k])
                assert same, (labels[b], k)
    assert {"dominant", "all_inf"} <= seen
    if version in ("barrage", "micro"):
        assert "single" in seen


# ---- float32 values -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("version", ["barrage", "standard", "micro", "fives"])
def test_float32_values_round_like_the_reference(version):
    """48 rounds with values 0.1 k and N(0, 2) (outside [-1, 1] too): W, a float32 sum leaf to root, bit for bit"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 3)

    def net_of(b, s, p, n_logits):
        logits, _ = net(s, p, n_logits)
        rng = np.random.default_rng(_key(s, p))
        return logits, f32(rng.integers(-25, 26) * 0.1) if b % 2 else f32(rng.standard_normal() * 2)

    _, tree, _ = _against_reference(e, version, dense, player, rows, 48, 2000, net_of=net_of)
    W = tree.value[:, 0].cpu().numpy()
    assert np.any(W * 1024 != np.round(W * 1024))  # sums that are not multiples of 1/16: the roundings were compared


# ---- deep lines -----------------------------------------------------------------------------------------------------
def _late_rows(version, k=6, near=12):
    """recorded states 1-3 plies before a recorded ending, and states within `near` plies of the turn limit"""
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    t = traj(version)
    S = t["states"]
    n = S.shape[0]
    max_turns = VERSION_CONFIGS[as_version(version)]["max_turns"]
    over = np.array([bool(data(S[i], OVER)) for i in range(n)])
    start = np.asarray(t["game_start"]).astype(bool)
    ends = [int(j - d) for j in np.flatnonzero(over) for d in (1, 2, 3)
            if j - d >= 0 and not over[j - d] and not start[j - d + 1:j + 1].any()]
    late = [i for i in range(n) if not over[i] and data(S[i], TURN) >= max_turns - near]
    return sorted(set(ends[::max(1, len(ends) // k)][:k] + late[::max(1, len(late) // k)][:k]))


@pytest.mark.parametrize("version,endings", [("micro", {"limit", "won"}), ("fives", {"limit", "won"}),
                                             ("tiny", {"won"}), ("short_barrage", {"limit"})])
def test_deep_lines_to_the_end_of_the_game(version, endings):
    """c_puct 0 and fpu -1: every round descends one ply deeper along the child-0 line until the game ends inside the
    tree (the turn limit, or a won game), 16 rounds from late recorded states.  Every round's leaf against the
    reference; the test asserts the depth and the endings it reached (Tiny's recorded games all end by capture long
    before its 100-ply limit, short_barrage's late states all run into it)"""
    e = _engine(version)
    rows = _late_rows(version)
    t = traj(version)
    dense = t["states"][rows].astype(np.int64)
    player = t["players"][rows].astype(np.int64)
    reached = set()
    deepest = [0]

    def after_round(r, tree, refs):
        node, kind = log[-1]
        parent = tree.parent.cpu().numpy()
        for b in range(len(rows)):
            d, x = 0, int(node[b])
            while x > 0:
                x, d = int(parent[b, x]), d + 1
            deepest[0] = max(deepest[0], d)
            if kind[b] == LEAF_OVER and d >= 1:
                reached.add("limit" if data(refs[b].states[int(node[b])][0], INVALID) else "won")

    log = []
    _against_reference(e, version, dense, player, rows, 16, 4000, c_puct=0.0, fpu=-1.0, after_round=after_round,
                       log=log)
    assert reached == endings and deepest[0] >= 9, (reached, deepest[0])


# ---- the score's extremes and ties ----------------------------------------------------------------------------------
def _score_rows(n, rng):
    """(label, N, W, P, c_puct, fpu) of the children of an expanded root: N int64, W and P float32"""
    M24 = (1 << 24) - 1
    out = []
    uniform = np.full(n, f32(1) / f32(n), f32)
    dirichlet = lambda: rng.dirichlet(np.full(n, 0.3)).astype(f32)  # noqa: E731
    N = rng.integers(0, 1 << 24, n)
    N[:3] = (M24, 0, M24)
    out.append(("large N", N, (N * rng.uniform(-1, 1, n)).astype(f32), dirichlet(), 1.25, 0.0))
    N = np.full(n, M24)
    W = np.where(np.arange(n) % 3 == 0, N, -N).astype(f32)
    W[1::7] = (N[1::7] * 0.37).astype(f32)
    out.append(("N 2^24-1, W +-N", N, W, dirichlet(), 2.5, 0.0))
    N = rng.integers(1, 1000, n)
    W = np.where(rng.random(n) < 0.5, N, -N).astype(f32)
    W[::5] = (N[::5] * f32(0.1)).astype(f32)
    out.append(("W +-N and fractions", N, W, uniform, 1.25, -0.5))
    P = np.zeros(n, f32)
    P[5], P[9], P[17], P[40] = f32(2.0 ** -149), f32(1e-40), f32(1), f32(2.0 ** -126)
    out.append(("P 0, subnormal, 1", np.zeros(n, np.int64), np.zeros(n, f32), P, 1.25, 0.0))
    N = rng.integers(0, 5, n)
    out.append(("P 0, subnormal, 1, visited", N, (N * rng.uniform(-1, 1, n)).astype(f32), P, 3.0, -1.0))
    N = rng.integers(1 << 16, 1 << 17, n)
    P = dirichlet()
    P[:3] = 0
    P = np.maximum(P, f32(1e-3)) * (np.arange(n) >= 3)
    P = P.astype(f32)
    out.append(("c_puct FLT_MAX: u = +inf", N, (N * rng.uniform(-1, 1, n)).astype(f32), P, FLT_MAX, 0.0))
    P2 = P.copy()
    P2[3:20] = f32(2.0 ** -140)
    out.append(("c_puct FLT_MAX, tiny P", N, (N * rng.uniform(-1, 1, n)).astype(f32), P2, FLT_MAX, -FLT_MAX))
    N = np.where(rng.random(n) < 0.5, 0, rng.integers(1, 50, n))
    N[:2] = (3, 0)
    W = (N * rng.uniform(-1, 1, n)).astype(f32)
    for fpu in (FLT_MAX, -FLT_MAX):
        out.append(("fpu %g" % fpu, N, W, dirichlet(), 1.25, fpu))
        out.append(("fpu %g, c_puct FLT_MAX" % fpu, N, W, dirichlet(), FLT_MAX, fpu))
    for tie in ([0, 31, 32, 33, 64], [31, 32, 33, 64], [32, 33, 64], [33, 64], [31, 64], [32, 64], [64], [31, 32]):
        P = np.full(n, f32(1e-3))
        P[tie] = f32(0.5)
        out.append(("tie %s" % tie, np.ones(n, np.int64), np.zeros(n, f32), P, 1.25, 0.0))
    return out


def test_score_extremes_and_ties():
    """select's arithmetic on the 83 children of an expanded Standard root, their N, W and P overwritten (select is a
    pure function of them): N up to 2^24 - 1 with the root's N = 1 + their sum, W at +-N and fractions, P 0, subnormal
    and 1, c_puct = FLT_MAX (u = +inf: the lowest child with P > 0), fpu = +-FLT_MAX, and exact ties at children 0, 31,
    32, 33 and 64 (two lanes, three 32-child passes).  The child taken is the first argmax of the numpy float32 score,
    both players to move"""
    e = _engine("standard")
    dense, player = _scouts()
    rng = np.random.default_rng(17)
    rows = _score_rows(83, rng)
    groups = {}
    for i, r in enumerate(rows):
        groups.setdefault((r[4], r[5]), []).append(i)
    checked = 0
    for (c_puct, fpu), idx in groups.items():
        B = 2 * len(idx)
        st = e.import_ref_state(torch.as_tensor(np.tile(dense, (len(idx), 1, 1, 1)), device="cuda"),
                                torch.as_tensor(np.tile(player, len(idx)).astype(np.int8), device="cuda"))
        tree = e.guided_tree(st, 200)
        leaves = e.guided_select(st, tree)
        e.guided_backup(tree, leaves, torch.zeros(B, *e.spatial_action_size, device="cuda"),
                        torch.zeros(B, device="cuda"))
        assert bool((tree.first_child[:, 0] == 1).all()) and bool((tree.n_children[:, 0] == 83).all())
        for k, i in enumerate(idx):
            _, N, W, P, _, _ = rows[i]
            for b in (2 * k, 2 * k + 1):
                tree.visits[b, 1:84] = torch.as_tensor(N.astype(np.int32), device="cuda")
                tree.value[b, 1:84] = torch.as_tensor(W, device="cuda")
                tree.prior[b, 1:84] = torch.as_tensor(P, device="cuda")
                tree.visits[b, 0] = int(1 + N.sum())
        node = e.guided_select(st, tree, c_puct=c_puct, fpu=fpu).node.cpu().numpy()
        for k, i in enumerate(idx):
            label, N, W, P, _, _ = rows[i]
            for b in (2 * k, 2 * k + 1):
                with np.errstate(over="ignore"):
                    s = scores(W, N, P, int(1 + N.sum()), int(player[b % 2]), c_puct, fpu)
                assert not np.isnan(s).any(), label
                assert int(node[b]) == 1 + int(np.argmax(s)), (label, int(player[b % 2]), int(node[b]) - 1,
                                                               int(np.argmax(s)))
                if label.startswith("tie"):
                    assert int(node[b]) - 1 == min(int(x) for x in label[5:-1].split(",")), label
                if label == "c_puct FLT_MAX: u = +inf":
                    assert np.isinf(s[3:]).all() and int(node[b]) == 1 + 3, label
                checked += 1
    assert checked == 2 * len(rows)


# ---- priors the caller rewrites -------------------------------------------------------------------------------------
@pytest.mark.parametrize("version", ["barrage", "micro", "standard2"])
def test_rewritten_priors(version):
    """after rounds 0 and 9 the root's children get 0.75 P + 0.25 Dirichlet(0.3) noise, mixed on the device with
    torch; the reference is given the same float32 priors, and the search still matches it round by round"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 3)
    rng = np.random.default_rng(23)
    changed = [0]

    def after_round(r, tree, refs):
        if r not in (0, 9):
            return
        for b, ref in enumerate(refs):
            f, n = int(tree.first_child[b, 0]), int(tree.n_children[b, 0])
            if f < 0:
                continue
            noise = torch.as_tensor(rng.dirichlet(np.full(n, 0.3)), dtype=torch.float32, device="cuda")
            old = tree.prior[b, f:f + n].clone()
            tree.prior[b, f:f + n] = 0.75 * old + 0.25 * noise
            changed[0] += int((tree.prior[b, f:f + n] != old).sum())
            ref.set_prior(f, tree.prior[b, f:f + n].cpu().numpy())

    _against_reference(e, version, dense, player, rows, 24, 2000, after_round=after_round)
    assert changed[0] > 0


# ---- root_stats of a guided tree ------------------------------------------------------------------------------------
@pytest.mark.parametrize("version", ["barrage", "micro"])
def test_root_stats_against_a_host_scatter(version):
    """visits and the values seen from the root's player to move at the entries of the root's moves, zero elsewhere,
    against a scatter of the tree (equal to the reference's) on the host"""
    e = _engine(version)
    dense, player, rows = _recorded(version, 4)

    def net_of(b, s, p, n_logits):
        logits, _ = net(s, p, n_logits)
        return logits, f32(np.random.default_rng(_key(s, p)).integers(-25, 26) * 0.1)

    st, tree, _ = _against_reference(e, version, dense, player, rows, 40, 2000, net_of=net_of)
    visits, values = tree.root_stats()
    R, C, A = e.spatial_action_size
    B = len(player)
    assert visits.shape == values.shape == (B, R, C, A)
    assert visits.dtype == torch.int32 and values.dtype == torch.float32
    mask = e.valid_mask(st).cpu().numpy().reshape(B, -1)
    mask[:, A - 1::A] = 0
    expanded = 0
    for b in range(B):
        h = _host(tree, b)
        wv, ww = np.zeros(R * C * A, np.int64), np.zeros(R * C * A, f32)
        kids = np.flatnonzero(h["parent"] == 0)
        wv[h["action"][kids]] = h["visits"][kids]
        ww[h["action"][kids]] = f32(player[b]) * h["value"][kids]
        assert np.array_equal(visits[b].reshape(-1).cpu().numpy(), wv), rows[b]
        assert np.array_equal(values[b].reshape(-1).cpu().numpy(), ww), rows[b]
        if kids.size:
            expanded += 1
            assert np.array_equal(np.flatnonzero(mask[b]), np.sort(h["action"][kids])), rows[b]
            assert int(wv.sum()) == 39
    assert expanded > 0
