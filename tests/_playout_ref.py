"""Reference of a random playout (sx_playout), on the reference's dense state layout.

Each ply draws the fused step's next-action word for the state before the ply (_sampler_ref.step_words: gid, turn,
episode, seed), picks the move with uniform_valid_ref over the oracle's mask of the player to move (maenv:447-497) and
plays it with the oracle's maenv:684-692 step.  A player whose mask holds only the noop entry without the game being
over is stuck: it plays the 1D noop (impl:912-920) and loses.  The playout stops when the oracle's game-over flag is set
or after max_plies plies."""
import numpy as np

from _sampler_ref import step_words, uniform_valid_ref

# scalar cells of the DATA layer (impl:136-142): [row, column]
TURN, OVER, WINNER, INVALID = (0, 0), (0, 1), (0, 2), (1, 1)
DATA = 5


def data(state, cell):
    return int(state[DATA][cell])


def playout_ref(orc, state, player, gid, episode, seed, max_plies):
    """(final dense state int64 [34, R, C], player to move, plies played, (over, winner, invalid))"""
    state = np.ascontiguousarray(state, dtype=np.int64).copy()
    player = int(player)
    plies = 0
    while plies < max_plies and not data(state, OVER):
        mask, _, _ = orc.current_obs(state, player, obs_mode=0)
        A = mask.shape[-1]
        word = step_words(np.array([gid]), data(state, TURN), episode, seed)
        a = int(uniform_valid_ref(mask.reshape(1, -1), word)[0])
        if a == A - 1:  # the noop entry is the whole mask: the player to move is stuck
            state, player = orc.base_env.get_next_state(state, player, orc.base_env.action_size - 1)
        else:
            state, player = orc.apply_spatial_action(state, player, a)
        plies += 1
    return state, player, plies, (data(state, OVER), data(state, WINNER), data(state, INVALID))
