"""Plain numpy reference of sx_sample_hidden_states (determinization of the opponent's hidden pieces), on the
reference's dense 34-layer state layout (no torch, no GPU).

Layers used (impl:16-60): 0 / 1 true rank of player +1 / -1, 2 obstacles, 3 / 4 partially observable rank (13 =
unknown), 8 + 12 * side + (code - 1) captured counts, 32 / 33 "still" (never moved).  Side 0 is player +1.

The contract (include/stratego_b200.h): the hidden cells of a game are the cells holding a piece of the viewer's
opponent that is not revealed (PO rank != true rank), on no obstacle.  Each hidden cell c of sample k of game b gets one
Philox4x32-10 block, key (seed lo, seed hi), counter (gid lo, gid hi, RNG_HIDDEN ^ draw, (k << 8) | c), gid = env_base +
b; words x and y are its sort keys.  The still hidden cells ordered by (x, c) take the immovable codes (flags, then
bombs) at ranks < I; the other hidden cells ordered by (y, c) take the movable codes in ascending order.  I > S (more
immovables than still hidden cells): the rows are copies and the status is 1.
"""
import numpy as np

from _sampler_ref import _key, philox4x32_10

M32 = np.uint64(0xFFFFFFFF)
RNG_HIDDEN = 0x48494444
FLAG, BOMB = 11, 12


def viewer_sides(player, viewer):
    """viewer side per game (0 = player +1): viewer None -> the player to move; else 1 -> +1, anything else -1"""
    src = np.asarray(player if viewer is None else viewer).reshape(-1)
    return np.where(src == 1, 0, 1).astype(np.int64)


def hidden_cells(dense, player, viewer):
    """(hidden [B, N] bool, still [B, N] bool, opp [B] side index of the viewer's opponent, true [B, N] their codes)"""
    dense = np.asarray(dense)
    B = dense.shape[0]
    flat = dense.reshape(B, dense.shape[1], -1).astype(np.int64)
    opp = 1 - viewer_sides(player, viewer)
    rows = np.arange(B)
    true = flat[rows, opp]
    po = flat[rows, 3 + opp]
    still = flat[rows, 32 + opp] != 0
    hidden = (true != 0) & (true <= BOMB) & (po != true) & (flat[:, 2] == 0)
    return hidden, still & hidden, opp, true


def code_counts(hidden, true):
    """[B, 13] number of hidden cells holding each code (column 0 unused)"""
    return np.stack([(hidden & (true == t)).sum(1) for t in range(13)], axis=1)


def _rank_in_row(row, k1, k2):
    """rank of every entry inside its row when the entries of a row are ordered by (k1, k2) ascending"""
    order = np.lexsort((k2, k1, row))
    rs = row[order]
    rank = np.empty(row.size, dtype=np.int64)
    rank[order] = np.arange(row.size) - np.searchsorted(rs, rs, side="left")
    return rank


def sample_hidden_ref(dense, player, viewer, n_samples, seed, draw=0, env_base=0, gids=None):
    """samples int64 [B * n_samples, 34, R, C] (row b * n_samples + k = sample k of game b) and status uint8 [B].
    gids (optional, [B]): the global id of each game instead of env_base + b (a scattered subset of a batch)"""
    dense = np.asarray(dense, dtype=np.int64)
    B, L, R, C = dense.shape
    K = int(n_samples)
    hidden, still, opp, true = hidden_cells(dense, player, viewer)
    cnt = code_counts(hidden, true)
    S = still.sum(1)
    n_flag = cnt[:, FLAG]
    I = cnt[:, FLAG] + cnt[:, BOMB]
    ok = I <= S
    out = np.repeat(dense, K, axis=0).reshape(B * K, L, R * C)
    eb, ec = np.nonzero(hidden & ok[:, None])
    es = still[eb, ec]
    E = eb.size
    if E == 0:
        return out.reshape(B * K, L, R, C), (~ok).astype(np.uint8)
    ek = np.repeat(np.arange(K, dtype=np.int64), E)
    eb, ec, es = np.tile(eb, K), np.tile(ec, K), np.tile(es, K)
    if gids is None:
        gid = eb.astype(np.uint64) + np.uint64(int(env_base) & (2 ** 64 - 1))  # wraps mod 2^64 like the kernel's
    else:
        gid = np.asarray(gids, dtype=np.uint64)[eb]
    k0, k1 = _key(seed)
    c2 = np.full(gid.shape, (RNG_HIDDEN ^ (int(draw) & 0xFFFFFFFF)) & 0xFFFFFFFF, dtype=np.uint64)
    x, y, _, _ = philox4x32_10(gid & M32, gid >> np.uint64(32), c2, (ek.astype(np.uint64) << np.uint64(8)) | ec.astype(np.uint64),
                               k0, k1)
    row = eb * K + ek
    code = np.zeros(row.size, dtype=np.int64)
    filled = np.zeros(row.size, dtype=bool)
    s = np.nonzero(es)[0]
    if s.size:
        r1 = _rank_in_row(row[s], x[s].astype(np.int64), ec[s])
        take = r1 < I[eb[s]]
        filled[s[take]] = True
        code[s[take]] = np.where(r1[take] < n_flag[eb[s[take]]], FLAG, BOMB)
    m = np.nonzero(~filled)[0]
    if m.size:
        r2 = _rank_in_row(row[m], y[m].astype(np.int64), ec[m])
        cum = np.cumsum(cnt[:, 1:11], axis=1)  # running count of the movable codes 1..10
        code[m] = 1 + (cum[eb[m]] <= r2[:, None]).sum(1)
    out[row, opp[eb], ec] = code
    return out.reshape(B * K, L, R, C), (~ok).astype(np.uint8)


def inferred_multiset(dense, player, viewer, piece_amounts):
    """[B, 13] what the viewer can infer of the opponent's unrevealed pieces: piece_amounts - captured - revealed alive"""
    dense = np.asarray(dense, dtype=np.int64)
    B = dense.shape[0]
    flat = dense.reshape(B, dense.shape[1], -1)
    opp = 1 - viewer_sides(player, viewer)
    rows = np.arange(B)
    true, po = flat[rows, opp], flat[rows, 3 + opp]
    out = np.zeros((B, 13), dtype=np.int64)
    for t in range(1, 13):
        captured = flat[rows, 8 + 12 * opp + (t - 1)].sum(1)
        revealed = ((true == t) & (po == t)).sum(1)
        out[:, t] = int(piece_amounts[t]) - captured - revealed
    return out
