"""The action samplers against the float64 reference of tests/_sampler_ref.py, draw for draw.

Every kernel draw is recomputed on the host from the same Philox counters (counter layouts: tests/_sampler_ref.py), so
a wrong counter, uniform, Gumbel transform, tie rule or log-sum-exp shows up as a mismatch in individual rows instead
of a drift a distribution test cannot see.

Policy samplers (sx_sample_logits, sx_sample_policy): for every row whose reference gap between the two best scores
exceeds tau, the kernel's action equals the reference action.  tau = 1e-4 + 2^-24 (|z_a - z_b| + 2 |z_a| + 2 |z_b|)
bounds what fp32 can move that gap (z = logit / T of the two best entries; derivation in gumbel_max_ref): the 1e-4
covers twice the Gumbel-transform error the probe below bounds (2e-5) plus the rounding of the scores.  Rows under tau
are excluded and must stay under 0.1 % of the rows, so the test cannot skip its way to a pass.

Log-probabilities are compared with float64 z_a - logsumexp(z over the valid entries) at the kernel's action a, with
|error| <= 1e-6 + 2 (m + 5) 2^-24 + 10 * 2^-24 * max |z_valid|:
- m + 5 roundings of a positive sum (m = ceil(valid / 32) terms per lane, 5 warp combines), and as many of the
  rescaling products, each a relative error of 2^-24 of the sum, i.e. an absolute error of 2^-24 in its log;
- 1e-6 for __expf (2 ulp relative per term) and __logf (2^-21.4 absolute on [0.5, 2], 3 ulp of |log| <= 10 beyond);
- 10 * 2^-24 * max|z|: z carries 2 roundings (1 / T and the product), which move z_a - lse by up to 4 of them;
  z - run_max another 2 inside the exponentials; the final run_max + log and z_a - (...) 2 more each.
Behaviour pinned for non-finite input: a valid logit of -inf has probability 0 and never breaks the log-probability;
if every valid logit is -inf the action is the lowest valid index and the log-probability is NaN (as torch's
log_softmax).  NaN and +inf logits at valid entries are undefined; invalid entries are never read (they hold NaN here).

The uniform draws (sx_sample_valid and the SX_SAMPLE_NEXT draw of the fused step) must equal the reference exactly."""
import numpy as np
import pytest
import torch

from _sampler_ref import gumbel64, gumbel_max_ref, policy_words, step_words, uniform64, uniform_valid_ref, valid_words

pytestmark = pytest.mark.gpu

DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
HIGH_SEED = 0x5EED_0000_0000_0002     # non-zero high key word (and the probe seed below)
HIGH_BASE = 2 ** 32 - 5               # rows straddle the high counter word
U24 = 2.0 ** -24


@pytest.fixture(scope="module")
def eng():
    from stratego_env_b200.config import BARRAGE_STRATEGO_CONFIG
    from stratego_env_b200.engine import StrategoEngine
    return StrategoEngine(BARRAGE_STRATEGO_CONFIG, device="cuda:0")


def _logprob_bound(z_valid_absmax, n_valid):
    m = np.ceil(np.asarray(n_valid) / 32.0)
    return 1e-6 + 2 * (m + 5) * U24 + 10 * U24 * z_valid_absmax


def _mask_view(mask_np, off):
    """the mask on the device at byte offset `off` of a 256-byte aligned buffer (a contiguous view)"""
    B, n = mask_np.shape
    buf = torch.zeros(B * n + 16, dtype=torch.uint8, device="cuda")
    view = buf[off:off + B * n].view(B, n)
    view.copy_(torch.from_numpy(mask_np))
    return view


def _tail_start(addr, n):
    """first index of a row's tail loop in sx_sample_logits_kernel (the mask row starts at byte address `addr`)"""
    head = min((4 - addr % 4) % 4, n)
    return head + ((n - head) >> 2 << 2)


def _row_masks(B, n, off, rng):
    """rows of every kind, cycled: fully dense (few), one valid entry at 0 / at n - 1 / in the tail loop, half dense,
    empty, and sparse (~1 %, at least 3 / n)"""
    mask = (rng.random((B, n)) < max(0.01, 3.0 / n)).astype(np.uint8)
    for r in range(B):
        kind = r % 16
        if kind == 0 and r < 64:
            mask[r] = 1
        elif kind in (1, 2, 3):
            mask[r] = 0
            ts = _tail_start(off + r * n, n)
            mask[r, {1: 0, 2: n - 1, 3: ts if ts < n else n - 1}[kind]] = 1
        elif kind == 4:
            mask[r] = rng.random(n) < 0.5
        elif kind == 5:
            mask[r] = 0
    return mask


def _draw_and_check(eng, logits, mask_np, off, T, env_base, seed, step, check_excluded=True):
    """runs sx_sample_logits and compares every row with the reference; returns the worst log-probability error
    relative to its bound and the number of excluded rows"""
    B, n = mask_np.shape
    mask = _mask_view(mask_np, off)
    dev = logits.to("cuda")
    actions, logp = eng.sample_logits(dev, mask, seed=seed, step=step, env_base=env_base, temperature=T,
                                      return_logprob=True)
    actions, logp = actions.cpu().numpy().astype(np.int64), logp.cpu().numpy().astype(np.float64)
    values = logits.to(torch.float64).numpy()
    gids = (np.arange(B, dtype=np.uint64) + np.uint64(env_base)) & np.uint64(2 ** 64 - 1)
    ref = gumbel_max_ref(values, mask_np, T, gids, seed, step)
    nvalid = mask_np.sum(1)
    empty = nvalid == 0
    assert (actions[empty] == -1).all()
    assert (actions[~empty] >= 0).all() and (mask_np[~empty, actions[~empty]] == 1).all()  # never an invalid entry
    decided = ref.gap > ref.tau
    bad = np.nonzero(decided & (actions != ref.action))[0]
    assert bad.size == 0, ("draws differ from the reference", bad[:8], actions[bad[:8]], ref.action[bad[:8]])
    excluded = int((~decided).sum())
    if check_excluded:
        assert excluded * 1000 <= B, (excluded, B)
    rows = np.nonzero(~empty)[0]
    z = values / T
    zabs = np.where(mask_np != 0, np.abs(z), 0.0)
    zabs[~np.isfinite(zabs)] = 0.0
    with np.errstate(invalid="ignore"):
        ref_lp = z[rows, actions[rows]] - ref.lse[rows]
    bound = _logprob_bound(zabs[rows].max(1), nvalid[rows])
    err = np.abs(logp[rows] - ref_lp)
    both_nan = np.isnan(ref_lp) & np.isnan(logp[rows])
    ok = both_nan | (err <= bound)
    assert ok.all(), ("log-probability", rows[~ok][:8], logp[rows][~ok][:8], ref_lp[~ok][:8], bound[~ok][:8])
    return float(np.max(np.where(both_nan, 0.0, err / bound), initial=0.0)), excluded


# (B, mask byte offset, T, env_base, seed, step)
LAUNCHES = [(1, 0, 1.0, 0, 5, 0),
            (7, 1, 0.05, HIGH_BASE, HIGH_SEED, 2 ** 32 - 1),
            (333, 2, 50.0, HIGH_BASE - 100, 7, 2 ** 32 - 2),
            (4096, 3, 1e-4, HIGH_BASE, HIGH_SEED, 12),
            (4096, 0, 1.0, 11, 2 ** 64 - 1, 2 ** 32 - 3)]


@pytest.mark.parametrize("n", [1, 2, 3, 5, 31, 33, 132, 1024 + 3, 2049, 3700, 12825])
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_sample_logits_draw_for_draw(eng, dtype, n):
    """every draw of sx_sample_logits equals the float64 Gumbel-max reference, over the head loop, the 8-word batches
    and the tail loop, mask rows at every address mod 4, rows straddling the high counter word, a seed with non-zero
    high bits, steps near 2^32 and temperatures 1e-4 .. 50"""
    rng = np.random.default_rng(n * 7 + len(dtype))
    g = torch.Generator().manual_seed(n)
    for B, off, T, env_base, seed, step in LAUNCHES:
        B = min(B, max(333, 2 ** 21 // n))           # bounds the host reference's time
        mask = _row_masks(B, n, off, rng)
        logits = (torch.randn(B, n, generator=g) * 3).to(DTYPES[dtype])
        logits[torch.from_numpy(mask == 0)] = float("nan")  # never read
        _draw_and_check(eng, logits, mask, off, T, env_base, seed, step)


@pytest.mark.parametrize("dtype", list(DTYPES))
@pytest.mark.parametrize("case", ["offset+1e3", "offset-1e3", "T0.05_randn10", "dense12825"])
def test_sample_logits_logprob_accuracy(eng, dtype, case):
    """log-probabilities against float64 where fp32 is stressed: a common offset of +-1e3 (the log-sum-exp must not
    lose it), T = 0.05 with randn*10 logits (|z| ~ 800) and dense 12 825-entry rows (~400 terms per lane)"""
    g = torch.Generator().manual_seed(len(case) * 31 + len(dtype))
    rng = np.random.default_rng(len(case))
    if case == "dense12825":
        B, n, T = 256, 12825, 1.0
        mask = np.ones((B, n), dtype=np.uint8)
        mask[B // 2:] = rng.random((B - B // 2, n)) < 0.9
        logits = torch.randn(B, n, generator=g) * 3
    else:
        B, n = 2048, 3700
        mask = (rng.random((B, n)) < 0.05).astype(np.uint8)
        mask[:, 5] = 1
        if case == "T0.05_randn10":
            T, logits = 0.05, torch.randn(B, n, generator=g) * 10
        else:
            T, logits = 1.0, torch.randn(B, n, generator=g) * 3 + (1e3 if case == "offset+1e3" else -1e3)
    worst = 0.0
    for off in range(4):
        w, _ = _draw_and_check(eng, logits.to(DTYPES[dtype]), mask, off, T, 3, 17 + off, off)
        worst = max(worst, w)
    print("%s %s: worst log-probability error / bound = %.3f" % (dtype, case, worst))


# ---- (b) the state-based sampler on real games ----------------------------------------------------------------------
# every launch_policy instantiation: K = 2 (N <= 64), K = 4 with and without compact movers (N = 100), K = 8 (N = 225)
POLICY_CASES = [("micro", None, -1), ("tiny", None, -1), ("fives", None, -1), ("medium", None, -1),
                ("octa_barrage", None, -1), ("barrage", "barrage", 0), ("barrage", "barrage", 1),
                ("standard", "standard", 0), ("standard", "standard", 1), ("standard2", None, -1)]


def _policy_engine(version, table):
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    from stratego_env_b200.engine import StrategoEngine, load_setup_table
    e = StrategoEngine(VERSION_CONFIGS[as_version(version)], device="cuda:0", p2_rot180=table is None)
    return e, (e.upload_setups(load_setup_table(table)) if table else None)


@pytest.mark.parametrize("version,table,compact", POLICY_CASES)
def test_sample_policy_draw_for_draw_on_real_states(version, table, compact):
    """sx_sample_policy on fresh, mid-game and finished games (no auto-reset: finished games keep their noop-only
    mask) equals the reference on the mover's-frame mask, with and without the log-probability"""
    e, setups = _policy_engine(version, table)
    if compact >= 0:
        e.set_tuning(compact_movers=compact)
    B, env_base, seed = 1000, HIGH_BASE - 500, HIGH_SEED
    R, C, A = e.spatial_action_size
    st = e.alloc_state(B)
    e.reset(st, seed=3, env_base=env_base, setups=setups, shuffle=setups is None)
    out = e.alloc_outputs(B, partial=False, full=False, mask=True, sample=True)
    e.observe(st, out=out, partial=False, full=False, mask=True)
    actions = e.sample_valid(out["valid_mask"], seed=3, env_base=env_base)
    g = torch.Generator().manual_seed(len(version))
    gids = np.arange(B, dtype=np.uint64) + np.uint64(env_base)
    finished = 0
    for s in range(61):
        if s in (0, 12, 60):
            mask_np = e.valid_mask(st).reshape(B, -1).cpu().numpy()
            dtype = torch.bfloat16 if s == 12 else torch.float32
            logits = (torch.randn(B, R * C * A, generator=g) * 2).to(dtype)
            T, step = (0.8, 2 ** 32 - 1 - s)
            a, lp = e.sample_policy(st, logits.cuda(), seed=seed, step=step, env_base=env_base, temperature=T,
                                    return_logprob=True)
            a_only = e.sample_policy(st, logits.cuda(), seed=seed, step=step, env_base=env_base, temperature=T)
            assert torch.equal(a, a_only)
            a, lp = a.cpu().numpy().astype(np.int64), lp.cpu().numpy().astype(np.float64)
            values = logits.to(torch.float64).numpy()
            ref = gumbel_max_ref(values, mask_np, T, gids, seed, step)
            decided = ref.gap > ref.tau
            assert (~decided).sum() * 1000 <= B
            bad = np.nonzero(decided & (a != ref.action))[0]
            assert bad.size == 0, (version, s, bad[:8], a[bad[:8]], ref.action[bad[:8]])
            z = values / T
            ref_lp = z[np.arange(B), a] - ref.lse
            zmax = np.where(mask_np != 0, np.abs(z), 0.0).max(1)
            bound = _logprob_bound(zmax, mask_np.sum(1))
            assert (np.abs(lp - ref_lp) <= bound).all(), float(np.abs(lp - ref_lp).max())
            noop_only = (mask_np.sum(1) == 1) & (mask_np[:, A - 1] == 1)
            assert (a[noop_only] == A - 1).all() and (lp[noop_only] == 0.0).all()
            finished = int(noop_only.sum())
        e.step_all(st, actions, out, env_base=env_base, auto_reset=False, sample_next=True, seed=3)
        actions = out["next_action"].clone()
    if version in ("micro", "tiny"):
        assert finished > 0


# ---- (d) -inf and extreme logits ------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_minus_inf_logits_keep_the_logprob_finite(eng, dtype):
    """valid entries with logit -inf placed where each lane starts (every index = 0 mod 4 of an aligned row, the
    entries lanes 0..k of the head loop visit first, the tail loop): the action is a finite-logit entry and the
    log-probability is finite and equals the reference.  Rows whose valid logits are ALL -inf draw their lowest valid
    index with a NaN log-probability, as torch.log_softmax gives."""
    B, n = 512, 256 + 3
    rng = np.random.default_rng(1)
    g = torch.Generator().manual_seed(2)
    logits = torch.randn(B, n, generator=g) * 2
    mask = (rng.random((B, n)) < 0.3).astype(np.uint8)
    mask[:, :4] = 1
    mask[:, n - 3:] = 1
    ninf = torch.zeros(B, n, dtype=torch.bool)
    ninf[0::4, 0::4] = True                       # each lane's first word starts with -inf
    ninf[1::4, :32] = True                        # the first 32 entries, i.e. every lane's first visit on sparse rows
    ninf[2::4, n - 3:] = True                     # tail loop
    ninf[3::8, :] = True                          # every valid logit -inf
    logits[ninf] = float("-inf")
    logits = logits.to(DTYPES[dtype])
    allinf = (ninf.numpy() | (mask == 0)).all(1)
    for off in (0, 1):
        m = _mask_view(mask, off)
        a, lp = eng.sample_logits(logits.cuda(), m, seed=4, step=9, temperature=1.0, return_logprob=True)
        a, lp = a.cpu().numpy().astype(np.int64), lp.cpu().numpy()
        assert np.isfinite(lp[~allinf]).all(), np.nonzero(~np.isfinite(lp) & ~allinf)[0][:8]
        assert np.isfinite(logits.float().numpy()[np.arange(B)[~allinf], a[~allinf]]).all()
        assert np.isnan(lp[allinf]).all()
        assert (a[allinf] == np.argmax(mask[allinf] != 0, axis=1)).all()
        _draw_and_check(eng, logits, mask, off, 1.0, 0, 4, 9)


def test_minus_inf_logits_through_the_state_sampler():
    """the same for sx_sample_policy: the even-ranked valid entries (each lane's first move when a game has more
    than 32 of them, every other lane's otherwise) get -inf"""
    e, setups = _policy_engine("barrage", "barrage")
    B = 512
    st = e.alloc_state(B)
    e.reset(st, seed=8, setups=setups)
    mask = e.valid_mask(st).reshape(B, -1)
    rank = torch.cumsum(mask.int(), 1) - 1
    logits = torch.randn(mask.shape, device="cuda")
    logits[(mask != 0) & (rank % 2 == 0)] = float("-inf")
    a, lp = e.sample_policy(st, logits, seed=8, step=1, return_logprob=True)
    assert torch.isfinite(lp).all()
    assert torch.isfinite(logits.gather(1, a.long()[:, None])).all()
    ref = gumbel_max_ref(logits.double().cpu().numpy(), mask.cpu().numpy(), 1.0, np.arange(B), 8, 1)
    lp_ref = logits.double().cpu().numpy()[np.arange(B), a.cpu().numpy()] - ref.lse
    assert np.allclose(lp.cpu().numpy(), lp_ref, rtol=0, atol=1e-5)
    assert np.array_equal(a.cpu().numpy()[ref.gap > ref.tau], ref.action[ref.gap > ref.tau])


def test_huge_negative_logits_and_subnormal_temperature(eng):
    """logits of -3e38 are finite: z must not become NaN; a subnormal temperature (1 / T = inf) is refused"""
    B, n = 256, 100
    rng = np.random.default_rng(3)
    mask = (rng.random((B, n)) < 0.2).astype(np.uint8)
    mask[:, 0] = 1
    logits = torch.randn(B, n) * 2
    logits[:, 0::3] = -3e38
    logits[B // 2:] = -3e38                        # every valid logit -3e38: uniform over the valid entries
    a, lp = eng.sample_logits(logits.cuda(), _mask_view(mask, 0), seed=2, step=2, return_logprob=True)
    lp = lp.cpu().numpy()
    assert np.isfinite(lp).all()
    nvalid = mask[B // 2:].sum(1)
    assert np.allclose(lp[B // 2:], -np.log(nvalid), rtol=0, atol=_logprob_bound(3e38, nvalid).max())
    # rows with finite logits besides: the reference decides the draw (the all -3e38 rows have tau ~ 1e32: excluded)
    _draw_and_check(eng, logits[: B // 2], mask[: B // 2], 0, 1.0, 0, 2, 2)
    for T in (1e-40, 0.0, -1.0):
        with pytest.raises(Exception, match="temperature"):
            eng.sample_logits(logits.cuda(), _mask_view(mask, 0), temperature=T)


# ---- (e) the Gumbel transform, measured ------------------------------------------------------------------------------
PROBE_STEP, PROBE_GIDS, PROBE_N = 0xFFFFFFF0, 2 ** 20, 16


def _ordered(x):
    b = np.asarray(x, dtype=np.float32).view(np.int32).astype(np.int64)
    return np.where(b >= 0, b, -(b & 0x7FFFFFFF))


def _from_ordered(k):
    k = np.asarray(k, dtype=np.int64)
    bits = np.where(k >= 0, k, (-k) | 0x80000000).astype(np.uint32)
    return bits.view(np.float32)


@pytest.fixture(scope="module")
def probes():
    return _find_probes()


def _find_probes():
    """(gid, probe entry i, partner entry j): probes whose k = word >> 9 is among the 64 largest and 64 smallest of
    2^23 (k = 2^23 - 1 and k = 0 included), and up to 45 per band of -log2(1 - u) = 1 .. 23; one probe per gid"""
    words = policy_words(np.arange(PROBE_GIDS, dtype=np.uint64)[None, :], np.arange(PROBE_N, dtype=np.uint64)[:, None],
                         HIGH_SEED, PROBE_STEP)                     # [entry, gid]
    k = (words >> np.uint32(9)).astype(np.int64)
    u = uniform64(words)
    assert (k == 0).any() and (k == 2 ** 23 - 1).any()
    ent, gid = np.nonzero((k < 64) | (k >= 2 ** 23 - 64))
    picks = [(gid, ent)]
    band = np.floor(-np.log2(1.0 - u)).astype(np.int64)
    for b in range(1, 24):
        e_b, g_b = np.nonzero(band == b)
        picks.append((g_b[:45], e_b[:45]))
    gid = np.concatenate([p[0] for p in picks])
    ent = np.concatenate([p[1] for p in picks])
    gid, first = np.unique(gid, return_index=True)                  # keeps the first pick of each gid
    ent = ent[first]
    mid = (u[:, gid] > 0.1) & (u[:, gid] < 0.9)
    mid[ent, np.arange(gid.size)] = False
    assert mid.any(0).all()
    partner = np.argmax(mid, axis=0)
    kk = k[ent, gid]
    assert (kk == 0).any() and (kk == 2 ** 23 - 1).any()
    return gid, ent, partner, words[ent, gid], words[partner, gid]


def test_gumbel_transform_matches_float64(eng, probes):
    """For each probe row (two valid entries: the probe i and a partner j with u_j in (0.1, 0.9), logit_j = 0,
    T = 1) bisect over the float32 logit x of entry i for the smallest x that makes i win: the kernel then says
    G_i - G_j = -x*.  Require |-x* - (G64_i - G64_j)| <= 2e-5 for every probe; the table printed is the measured
    maximum error per band of -log2(1 - u_i) (row 'k<64': the 64 smallest k)."""
    gid, ent, partner, w_i, w_j = probes
    P = gid.size
    mask = torch.zeros(PROBE_GIDS, PROBE_N, dtype=torch.uint8, device="cuda")
    gi, ei, pj = (torch.from_numpy(v.astype(np.int64)).cuda() for v in (gid, ent, partner))
    mask[gi, ei] = 1
    mask[gi, pj] = 1
    logits = torch.zeros(PROBE_GIDS, PROBE_N, device="cuda")

    def wins(x):
        logits[gi, ei] = torch.from_numpy(x).cuda()
        a = eng.sample_logits(logits, mask, seed=HIGH_SEED, step=PROBE_STEP, env_base=0, temperature=1.0)
        return (a[gi] == ei.int()).cpu().numpy()

    lo, hi = np.full(P, _ordered(-64.0)), np.full(P, _ordered(64.0))
    assert not wins(_from_ordered(lo)).any() and wins(_from_ordered(hi)).all()
    while (hi - lo > 1).any():
        mid = (lo + hi) // 2
        w = wins(_from_ordered(mid))
        hi = np.where(w, mid, hi)
        lo = np.where(w, lo, mid)
    measured = -_from_ordered(hi).astype(np.float64)
    expect = gumbel64(w_i) - gumbel64(w_j)
    err = np.abs(measured - expect)
    u = uniform64(w_i)
    k = (w_i >> np.uint32(9)).astype(np.int64)
    band = np.where(k < 64, 0, np.floor(-np.log2(1.0 - u))).astype(np.int64)
    print("\nGumbel transform G_i - G_j, kernel vs float64 (%d probes)" % P)
    print("%-10s %6s %12s" % ("band", "probes", "max |err|"))
    for b in np.unique(band):
        sel = band == b
        print("%-10s %6d %12.3e" % ("k<64" if b == 0 else "-log2(1-u)=%d" % b if b < 24 else "k=2^23-1",
                                    int(sel.sum()), float(err[sel].max())))
    worst = np.argsort(-err)[:5]
    assert (err <= 2e-5).all(), ("Gumbel transform error", [(int(k[i]), float(err[i])) for i in worst])


# ---- (f) the uniform draws -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("mask_len", [1, 31, 32, 33, 3700])
def test_sample_valid_equals_reference(eng, mask_len):
    B = 999
    rng = np.random.default_rng(mask_len)
    mask = (rng.random((B, mask_len)) < rng.random((B, 1))).astype(np.uint8)
    mask[0::7] = 0                                 # empty rows: -1
    one = np.arange(B)[3::7]
    mask[one] = 0
    mask[one, rng.integers(0, mask_len, one.size)] = 1  # single-entry rows
    for env_base, seed, step in ((0, 1, 0), (HIGH_BASE - 400, HIGH_SEED, 2 ** 32 - 1)):
        got = eng.sample_valid(torch.from_numpy(mask).cuda(), seed=seed, step=step, env_base=env_base)
        gids = np.arange(B, dtype=np.uint64) + np.uint64(env_base)
        ref = uniform_valid_ref(mask, valid_words(gids, seed, step))
        assert np.array_equal(got.cpu().numpy(), ref)


@pytest.mark.parametrize("auto_reset", [False, True])
@pytest.mark.parametrize("version,table,baseline", [("barrage", "barrage", True), ("micro", None, False),
                                                    ("tiny", None, False)])
def test_step_next_action_equals_reference(version, table, baseline, auto_reset):
    """next_action of step_all(sample_next=True) is the uniform draw over the post-step mask keyed by the post-step
    aux (turn, episode), in the warp-level kernel and the thread-per-game kernel, with and without auto-reset"""
    e, setups = _policy_engine(version, table)
    B, env_base, seed = 700, HIGH_BASE - 300, HIGH_SEED
    assert e.launch_info(partial=True, mask=True)["thread_per_game"] == (0 if version == "barrage" else 1)
    st = e.alloc_state(B)
    e.reset(st, seed=seed, env_base=env_base, setups=setups, shuffle=setups is None)
    out = e.alloc_outputs(B, partial=True, full=False, mask=True, sample=True)
    e.observe(st, out=out)
    actions = e.sample_valid(out["valid_mask"], seed=seed, env_base=env_base)
    gids = np.arange(B, dtype=np.uint64) + np.uint64(env_base)
    done_seen = 0
    for s in range(45):
        e.step_all(st, actions, out, env_base=env_base, auto_reset=auto_reset, sample_next=True, seed=seed,
                   setups=setups, shuffle=setups is None, baseline_kernel=baseline)
        aux = st.aux.contiguous().view(torch.int32).cpu().numpy().view(np.uint32)  # [B, 4] aux words
        mask = out["valid_mask"].reshape(B, -1).cpu().numpy()
        ref = uniform_valid_ref(mask, step_words(gids, aux[:, 0] & 0xFFFF, aux[:, 3], seed))
        got = out["next_action"].cpu().numpy()
        bad = np.nonzero(got != ref)[0]
        assert bad.size == 0, (s, bad[:8], got[bad[:8]], ref[bad[:8]])
        done_seen += int(out["done"].sum())
        actions = out["next_action"].clone()
    if version != "barrage":
        assert done_seen > 0
