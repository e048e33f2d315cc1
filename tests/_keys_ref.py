"""Plain numpy reference of sx_state_keys (64-bit Zobrist keys of positions and of information sets), on the reference's
dense 34-layer state layout (no torch, no GPU).

The contract (include/stratego_b200.h): the state key of (dense, player) is the XOR of Z(c, l, x) over every non-zero
entry x at (layer l, cell c) of layers 0-1 and 3-33, and Z(0, 34, player).  The information-set key for a viewer
replaces, on the viewer's hidden cells (_hidden_ref.hidden_cells), the opponent's true rank in layer opp with the PO
entry of layer 3 + opp, and adds Z(0, 35, viewer).  Z(c, l, x) = w0 | w1 << 32, (w0, w1) the first two words of
Philox4x32-10 with key (KEY_LO, KEY_HI) and counter (c, l, uint32(x), RNG_KEYS).
"""
import numpy as np

from _hidden_ref import hidden_cells, viewer_sides
from _sampler_ref import philox4x32_10

RNG_KEYS = 0x4B455953
KEY_LO, KEY_HI = 0x53545241, 0x5445474F
LAYER_PLAYER, LAYER_VIEWER = 34, 35
OBSTACLES = 2


def zobrist(cell, layer, value):
    """Z(c, l, x) as uint64 (arrays broadcast; x may be negative: it enters as uint32)"""
    cell, layer, value = np.broadcast_arrays(*(np.asarray(v, dtype=np.int64) for v in (cell, layer, value)))
    w0, w1, _, _ = philox4x32_10(cell, layer, value & 0xFFFFFFFF, np.full(cell.shape, RNG_KEYS, dtype=np.int64),
                                 KEY_LO, KEY_HI)
    return w0.astype(np.uint64) | (w1.astype(np.uint64) << np.uint64(32))


def _side_value(side):
    return np.where(np.asarray(side) == 0, 1, -1)


def state_keys_ref(dense, player, info_set=False, viewer=None):
    """uint64 [B] keys of the dense states int64 [B, 34, R, C] with player to move player [B] (+1 / -1).
    info_set=True: the information-set key for viewer [B] (1 = player +1, anything else -1; None = the player to move)"""
    dense = np.asarray(dense, dtype=np.int64)
    player = np.asarray(player).reshape(-1).astype(np.int64)
    B = dense.shape[0]
    flat = dense.reshape(B, dense.shape[1], -1).copy()
    if info_set:
        hidden, _, opp, _ = hidden_cells(dense, player, viewer)
        rows = np.arange(B)
        flat[rows, opp] = np.where(hidden, flat[rows, 3 + opp], flat[rows, opp])
    flat[:, OBSTACLES] = 0
    b, l, c = np.nonzero(flat)
    keys = np.zeros(B, dtype=np.uint64)
    np.bitwise_xor.at(keys, b, zobrist(c, l, flat[b, l, c]))
    keys ^= zobrist(0, LAYER_PLAYER, np.where(player == 1, 1, -1))
    if info_set:
        keys ^= zobrist(0, LAYER_VIEWER, _side_value(viewer_sides(player, viewer)))
    return keys
