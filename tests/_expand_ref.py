"""Reference for the children of a game (sx_count_moves / sx_expand_moves), on the reference's dense state layout.

The action list is the valid-action mask of the player to move (the oracle's restatement of maenv:447-497) without the
noop channel A-1, in ascending flat spatial index; each child is the oracle's maenv:684-692 step of that action: a dense
state and the next player."""
import numpy as np


def logic(version):
    from oracle.binding import OracleEnvLogic
    from stratego_env_b200.config import VERSION_CONFIGS, as_version
    cfg = VERSION_CONFIGS[as_version(version)]
    return OracleEnvLogic(cfg["rows"], cfg["columns"], cfg["piece_amounts"])


def action_list(orc, state, player):
    """int64 [n]: flat spatial indices of the legal moves of `player`, ascending (empty for a finished game or a stuck
    player, whose mask holds the noop entry only)"""
    mask, _, _ = orc.current_obs(np.ascontiguousarray(state, dtype=np.int64), int(player), obs_mode=0)
    A = mask.shape[-1]
    idx = np.flatnonzero(mask.reshape(-1))
    return idx[idx % A != A - 1]


def expand_ref(orc, state, player):
    """(actions int64 [n], children int64 [n, 34, R, C], next players int64 [n])"""
    state = np.ascontiguousarray(state, dtype=np.int64)
    acts = action_list(orc, state, player)
    kids = [orc.apply_spatial_action(state, int(player), int(a)) for a in acts]
    R, C = state.shape[1:]
    if not kids:
        return acts, np.zeros((0, 34, R, C), np.int64), np.zeros(0, np.int64)
    return acts, np.stack([k[0] for k in kids]), np.array([k[1] for k in kids], np.int64)
