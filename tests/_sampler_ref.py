"""Plain numpy / float64 reference of the action samplers (no torch, no GPU).

Counter layouts, as the kernels build them (gid = env_base + row, key = (seed lo, seed hi)):
- policy samplers, sx_policy.cu (sx_sample_logits_kernel, sx_sample_policy_kernel):
  counter (gid lo, gid hi, RNG_POLICY ^ step, entry)
- sx_sample_valid, sx_kernels.cu (sx_sample_kernel): counter (gid lo, gid hi, RNG_SAMPLE, step)
- the draw inside the fused step (SX_SAMPLE_NEXT), sx_kernels.cu (both step kernels):
  counter (gid lo, gid hi, RNG_SAMPLE ^ turn, episode), with turn = aux word 0 & 0xffff and episode = aux word 3 of the
  state the step wrote (aux_pack, sx_device.cuh)
Only the first output word of each Philox block is used.
"""
import numpy as np

M32 = np.uint64(0xFFFFFFFF)
RNG_POLICY = 0x504F4C59
RNG_SAMPLE = 0x53414D50


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11; Random123) over uint32 arrays; returns the four output words (uint32).
    The key is bumped after every round, like philox4x32_10 in sx_device.cuh."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & M32 for c in (c0, c1, c2, c3))
    k0, k1 = np.asarray(k0, dtype=np.uint64) & M32, np.asarray(k1, dtype=np.uint64) & M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & M32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & M32
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def _key(seed):
    seed = int(seed) & (2 ** 64 - 1)
    return seed & 0xFFFFFFFF, seed >> 32


def policy_words(gid, entry, seed, step):
    """first Philox word of the policy samplers' draw for (gid, entry) (arrays broadcast)"""
    gid = np.asarray(gid, dtype=np.uint64)
    k0, k1 = _key(seed)
    c2 = np.uint64((RNG_POLICY ^ (int(step) & 0xFFFFFFFF)) & 0xFFFFFFFF)
    entry = np.asarray(entry, dtype=np.uint64)
    gid, entry = np.broadcast_arrays(gid, entry)
    return philox4x32_10(gid & M32, gid >> np.uint64(32), np.full(gid.shape, c2), entry, k0, k1)[0]


def valid_words(gid, seed, step):
    """first Philox word of sx_sample_valid's draw for each gid"""
    gid = np.asarray(gid, dtype=np.uint64)
    k0, k1 = _key(seed)
    return philox4x32_10(gid & M32, gid >> np.uint64(32), np.full(gid.shape, RNG_SAMPLE, dtype=np.uint64),
                         np.full(gid.shape, int(step) & 0xFFFFFFFF, dtype=np.uint64), k0, k1)[0]


def step_words(gid, turn, episode, seed):
    """first Philox word of the fused step's next-action draw (turn, episode: the post-step aux fields)"""
    gid = np.asarray(gid, dtype=np.uint64)
    k0, k1 = _key(seed)
    c2 = np.uint64(RNG_SAMPLE) ^ (np.asarray(turn, dtype=np.uint64) & np.uint64(0xFFFF))
    return philox4x32_10(gid & M32, gid >> np.uint64(32), c2, np.asarray(episode, dtype=np.uint64), k0, k1)[0]


def uniform64(word):
    """u = ((word >> 9) + 0.5) / 2^23: the kernels' uniform, exact in float64 (and in float32)"""
    return ((np.asarray(word, dtype=np.uint32) >> np.uint32(9)).astype(np.float64) + 0.5) / 2.0 ** 23


def gumbel64(word):
    """the Gumbel variate G = -log(-log(u)) the kernels add to z = logit / T, in float64"""
    return -np.log(-np.log(uniform64(word)))


class GumbelMaxRef:
    """Reference draw of one batch of rows: fields action [B] (int64, -1 for an empty row), gap [B] (top score minus
    the runner-up, +inf with fewer than two valid entries or a -inf runner-up), tau [B] (the row's fp32 error bound on
    that gap, see gumbel_max_ref) and lse [B] (float64 log-sum-exp of z over the valid entries)."""

    def __init__(self, action, gap, tau, lse):
        self.action, self.gap, self.tau, self.lse = action, gap, tau, lse


def gumbel_max_ref(logits, mask, temperature, gids, seed, step, g_err=2e-5):
    """Gumbel-max draw over mask != 0 from logits [B, n] (the values the kernel reads, any float dtype), in float64:
    action = argmax over valid i of z_i + G_i with z = logits / T and G = gumbel64(policy_words(gid, i)); ties go to
    the lowest index.  Invalid entries are never read (they may hold anything).  A row whose valid logits are all -inf
    draws its lowest valid index.

    tau bounds how far the fp32 kernel can move the gap between the two best scores a and b.  With u = 2^-24:
    z_k = l_k * fl(1/T) carries the relative error of 1/T (u) and of the product (u); the score z_k + G_k is rounded
    once more (u |z_k + G_k|, |G_k| <= 17); G_k itself is off by at most g_err (the Gumbel probe measures it).  Summed
    over both entries: |error| <= 2 g_err + u (|z_a - z_b| + 2 |z_a| + 2 |z_b| + 34) + ... , so
    tau = 1e-4 + 2^-24 (|z_a - z_b| + 2 |z_a| + 2 |z_b|), i.e. 1e-4 absolute on top of 2 g_err = 4e-5."""
    logits = np.asarray(logits, dtype=np.float64)
    mask = np.asarray(mask) != 0
    B, n = logits.shape
    gids = np.asarray(gids, dtype=np.uint64).reshape(B)
    rows, cols = np.nonzero(mask)
    z = logits[rows, cols] / float(temperature)
    g = gumbel64(policy_words(gids[rows], cols, seed, step))
    with np.errstate(invalid="ignore"):
        score = z + g
    action = np.full(B, -1, dtype=np.int64)
    gap = np.full(B, np.inf)
    tau = np.full(B, 1e-4)
    lse = np.full(B, -np.inf)
    if rows.size == 0:
        return GumbelMaxRef(action, gap, tau, lse)
    # per row: sort the valid entries by (score descending, index ascending); np.lexsort sorts by the last key first
    order = np.lexsort((cols, -score, rows))
    r_sorted = rows[order]
    first = np.ones(order.size, dtype=bool)
    first[1:] = r_sorted[1:] != r_sorted[:-1]
    top = order[first]
    action[rows[top]] = cols[top]
    # runner-up: the next entry of the same row in that order
    nxt = np.nonzero(first)[0] + 1
    has2 = nxt < order.size
    has2[has2] = r_sorted[nxt[has2]] == r_sorted[nxt[has2] - 1]
    a_i, b_i = top[has2], order[nxt[has2]]
    r2 = rows[a_i]
    with np.errstate(invalid="ignore"):
        gap[r2] = score[a_i] - score[b_i]
        za, zb = z[a_i], z[b_i]
        tau[r2] = 1e-4 + 2.0 ** -24 * (np.abs(za - zb) + 2 * np.abs(za) + 2 * np.abs(zb))
    gap[np.isnan(gap)] = np.inf   # both best scores -inf: the tie rule decides exactly, nothing to exclude
    tau[~np.isfinite(tau)] = 0.0  # a -inf runner-up: any finite best wins outright
    # log-sum-exp over the valid entries of each row
    zmax = np.full(B, -np.inf)
    np.maximum.at(zmax, rows, z)
    shift = np.where(np.isfinite(zmax), zmax, 0.0)
    s = np.zeros(B)
    with np.errstate(invalid="ignore"):
        np.add.at(s, rows, np.exp(z - shift[rows]))
    with np.errstate(divide="ignore"):
        lse = np.where(s > 0, shift + np.log(s), -np.inf)
    return GumbelMaxRef(action, gap, tau, lse)


def uniform_valid_ref(mask, word, empty=-1):
    """The t-th set entry of each mask row in flat order, t = (word * total) >> 32; `empty` where a row has no set
    entry (sx_sample_valid returns -1; the fused step draws from the mover's moves and writes the noop entry A - 1
    when there are none, whose mask row then holds that entry alone)."""
    mask = np.asarray(mask).reshape(len(word), -1) != 0
    total = mask.sum(axis=1).astype(np.uint64)
    t = (np.asarray(word, dtype=np.uint64) * total) >> np.uint64(32)
    csum = np.cumsum(mask, axis=1)
    out = np.full(mask.shape[0], empty, dtype=np.int64)
    ok = total > 0
    # the first index whose running count exceeds t
    out[ok] = np.argmax(csum[ok] > t[ok, None].astype(np.int64), axis=1)
    return out
