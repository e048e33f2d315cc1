/*
 * stratego_b200.h -- C ABI of the B200-native batched Stratego engine.
 *
 * This is the drop-in boundary for the hot path of JBLanier/stratego_env: the per-step game logic
 * of stratego_env/game (valid-action mask, move/combat resolution, observation rendering,
 * auto-reset).  The reference has no FFI of its own -- the path sits behind two plain-Python
 * interfaces, StrategoProceduralEnv (stratego_env/game/stratego_procedural_env.py:20-173, "penv")
 * and StrategoMultiAgentEnv (stratego_env/stratego_multiagent_env.py:316-834, "maenv") -- so each
 * entry point below cites the reference function(s) it replaces ("impl" =
 * stratego_env/game/stratego_procedural_impl.py).  INTEGRATION.md shows the ctypes binding.
 *
 * Conventions
 *   - Every `*_d` / sx_state pointer is a DEVICE pointer owned by the caller (torch tensors in the
 *     Python host layer).  The library never allocates or frees caller-visible memory, except through
 *     sx_device_alloc / sx_device_free and in the sx_host_env convenience object at the bottom, which
 *     owns its own device buffers.
 *   - Every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without
 *     synchronising.  Return value: 0 = ok, negative = error (sx_last_error() has the text).
 *   - Games are independent: `num_envs` games, game b uses row b of every tensor.
 *   - "player" is +1 (moves first, owns rows 0..) or -1, as in the reference.
 *   - Frames: observations, spatial masks and spatial actions are in the frame of the player they
 *     are for (player -1 sees the board rotated 180 degrees, impl:646-675); device state and 1D
 *     actions are in the absolute frame, as in the reference.
 */
#ifndef STRATEGO_B200_H
#define STRATEGO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SX_PO_CHANNELS 67 /* impl:1332 */
#define SX_FO_CHANNELS 79 /* impl:1227 */
#define SX_PO_CHANNELS_ORIGINAL 32 /* impl:1148, deprecated obs_channel_mode='original' */
#define SX_FO_CHANNELS_ORIGINAL 33 /* impl:1070 */
#define SX_NUM_STATE_LAYERS 34 /* impl:109 */
#define SX_MAX_CAPTURE_COUNT 8

typedef struct sx_config sx_config; /* opaque, host-side */

/* Game variant description (one of the reference's config.py:3-313 dicts plus the host-computed
 * normalisation tables, maenv:202-313, 387-396, 499-508).  All pointers are HOST pointers and are
 * copied. */
typedef struct {
    int32_t rows, cols;           /* 3..15 each */
    int32_t max_turns;            /* 1..65535 */
    int32_t usable_rows;          /* initial_state_usable_rows */
    int32_t piece_amounts[13];    /* per piece code 1..12 (0 unused) */
    const uint8_t *obstacles;     /* [rows*cols] 0/1 */
    const float *captured_lut;    /* [12][SX_MAX_CAPTURE_COUNT+1] normalised captured-count values */
    const float *recent_lut;      /* [5] normalised recent-move codes -3..+1 */
    const float *unit_lut;        /* [2] normalised 0 and 1 of the one-hot/obstacle/still channels */
    int32_t p2_rot180;            /* setup rows for player -1 are rotated 180 deg (util:33-53) instead of
                                     row-mirrored (human tables, util:241-275) */
    int32_t capture_capacity;     /* capture-list entries per game; 0 = 2 * pieces per side (enough for any game
                                     played from this variant's setups); the stateless facade passes rows*cols */
    int32_t obs_channel_mode;     /* SX_CHANNELS_EXTENDED (67 / 79 one-hot channels, impl:1232-1397) or
                                     SX_CHANNELS_ORIGINAL (deprecated 32 / 33 raw-value channels, impl:1048-1197;
                                     env_config['obs_channel_mode'], maenv:370-375).  In the original mode unit_lut
                                     holds the normalised 0 and 1 of the obstacle / still channels (hi 2, lo 0) and
                                     captured_lut the hi-2 variant (maenv:87-199) */
    const float *rank_lut;        /* [14] original mode: normalised true rank 0..12 (entry 13 unused) */
    const float *po_rank_lut;     /* [14] original mode: normalised partially observable rank 0..13 */
    int32_t obs_dtype;            /* element type of every observation output (partial / full, terminal, sx_observe,
                                     sx_host_env): SX_DTYPE_F32 (0, the default of a zeroed descriptor), SX_DTYPE_BF16 or
                                     SX_DTYPE_F16.  A 16-bit element is the round-to-nearest-even conversion of the
                                     float32 the SX_DTYPE_F32 configuration writes for the same state */
} sx_config_desc;

enum { SX_CHANNELS_EXTENDED = 0, SX_CHANNELS_ORIGINAL = 1 };
enum { SX_DTYPE_F32 = 0, SX_DTYPE_BF16 = 1, SX_DTYPE_F16 = 2 }; /* obs_dtype; also the logits types of the samplers */

/* Byte/element strides of the device tensors for one variant. */
typedef struct {
    int32_t rows, cols, cells;
    int32_t spatial_channels;     /* A = 2(R-1)+2(C-1)+1, impl:258-259 */
    int32_t spatial_actions;      /* R*C*A = bytes of one uint8 spatial mask */
    int32_t action_size;          /* R*C*(R+C)+1, impl:253-254 */
    int32_t board_stride;         /* uint8 per env (cells rounded up to 16) */
    int32_t aux_stride;           /* int16 per env (= 8) */
    int32_t captured_stride;      /* uint16 per env */
    int32_t po_floats, fo_floats; /* elements per env of each observation (float32 or 16-bit: obs_elem_bytes) */
    int32_t setup_len;            /* usable_rows*cols bytes per setup-table row */
    int32_t pieces_per_side;
    int32_t po_channels, fo_channels; /* 67 / 79, or 32 / 33 in the original channel mode */
    int32_t obs_elem_bytes;       /* 4 (SX_DTYPE_F32) or 2 (SX_DTYPE_BF16 / SX_DTYPE_F16) */
} sx_layout;

/* Compact struct-of-arrays device state (DESIGN.md "State layout"). */
typedef struct {
    uint8_t *board;     /* [num_envs][board_stride] one packed byte per cell */
    int16_t *aux;       /* [num_envs][8] turn, max_turns, flags, recent moves, episode counter */
    uint16_t *captured; /* [num_envs][captured_stride] (cell, owner, type, count) capture entries */
} sx_state;

/* Per-step outputs; any pointer may be NULL to skip that output.  The four observation pointers are typed float, but
 * their elements are of the configuration's obs_dtype (float32, or bfloat16 / float16: 2 bytes each). */
typedef struct {
    float *partial_obs;      /* [num_envs][R][C][67 | 32] obs_dtype, maenv:461-475 (normalised) */
    float *full_obs;         /* [num_envs][R][C][79 | 33] obs_dtype, maenv:480-492 (normalised) */
    uint8_t *valid_mask;     /* [num_envs][R][C][A] uint8 0/1, maenv:454 / impl:400-517 */
    float *reward;           /* [num_envs] player +1's reward when the game ended this step, else 0
                                (maenv:777-801: +-1, or 0 for an invalid ending) */
    uint8_t *done;           /* [num_envs] game ended this step (maenv:772) */
    int8_t *winner;          /* [num_envs] +1 / -1 / 0, state[5,0,2] (impl:140) of the ended game */
    uint8_t *ending_invalid; /* [num_envs] impl:846-849 */
    uint8_t *illegal;        /* [num_envs] 1 = action rejected, game left untouched (ValueError, impl:899-902);
                                2 = the game's capture list overflowed: the compact state no longer matches what the
                                reference's dense counters (impl:999-1009) would hold (sticky until the game is re-set;
                                cannot happen in games played from the variant's own setups) */
    int8_t *player;          /* [num_envs] player the returned mask/obs are for (= player to move) */
    int32_t *next_action;    /* [num_envs] uniformly sampled valid spatial action for `player`
                                (replaces maenv:830-834), written when SX_SAMPLE_NEXT is set */
    /* maenv:772-773: when a game ends, BOTH players get their observation of the final position.  With SX_AUTO_RESET the
     * regular outputs already show the next game, so these optional side buffers receive the terminal observations:
     * [num_envs][2][R][C][channels], index 0 = player +1's view, 1 = player -1's; only rows of games with done = 1 are
     * written.  (The terminal valid-action mask is the lone noop entry [0,0,A-1] for both players, impl:414 / 514-515.)
     * Each needs its regular counterpart (partial_obs / full_obs) to be requested in the same call. */
    float *terminal_partial_obs;
    float *terminal_full_obs;
} sx_outputs;

enum {
    SX_ACTION_SPATIAL = 0, /* flat index into (R,C,A) in the mover's frame, as fed to maenv.step (maenv:685) */
    SX_ACTION_1D = 1       /* absolute 1D index incl. trailing noop, as fed to penv.get_next_state (penv:148) */
};

enum {
    SX_AUTO_RESET = 1,          /* games that end are re-set in the same call; outputs show the new game */
    SX_SAMPLE_NEXT = 2,         /* also draw a uniformly random valid action into outputs.next_action */
    SX_ALLOW_OSCILLATION = 4,   /* allow_piece_oscillation=True (impl:771-777) */
    SX_RESET_RANDOM_SHUFFLE = 8, /* (re)sets draw setups by shuffling the pieces (util:13-30) instead of a table */
    SX_SAME_SETUP = 32,         /* same_start_pos_everytime (maenv:352-354): every game of an env starts from the setup
                                   its first draw produced */
    SX_REPEAT_OTHER_SIDE = 64,  /* repeat_games_from_other_side (maenv:530-534): every second game of an env repeats the
                                   previous game's initial position as player -1 sees it (impl:646-675), player -1 first */
    SX_KERNEL_BASELINE = 16     /* run the general warp-per-game kernel even where a specialised one is eligible (the
                                   thread-per-game kernel of the <= 16-cell boards).  Results are identical by
                                   contract; the cross-kernel parity tests use it */
};

const char *sx_last_error(void);
int sx_version(void);

int sx_config_create(const sx_config_desc *desc, sx_config **out);
void sx_config_destroy(sx_config *cfg);
int sx_config_layout(const sx_config *cfg, sx_layout *out);

/* Launch tuning of the warp-level kernel; a development aid (tools/sweep_tuning.py times the library with it).
 * Every setting gives bit-identical results -- only the speed changes.  -1 keeps the built-in choice.
 *   warps_per_block  resident warps per SM (0 = built-in again)
 *   issue_point      where a game's background copy is handed to the TMA engine: 0 right before the sparse entries,
 *                    1 after the outcome of the move is known, 2 at the top of the game
 *   compact_movers   0 / 1: move generation hands the movable pieces to lanes instead of walking cells (10x10 class) */
int sx_config_set_tuning(sx_config *cfg, int32_t warps_per_block, int32_t issue_point, int32_t compact_movers);

/* Curriculum start states (curriculum_start_states_path, maenv:341-351 / 519-527, util:373-387): from now on every
 * (re)set of a game with this configuration -- sx_reset and the auto-reset inside sx_step_all -- copies a uniformly
 * drawn entry of `table` (n_states compact states, e.g. made with sx_import_ref_state from the file's dense states)
 * instead of dealing setups; the turn counter restarts at 0 with the configured max_turns (util:382-383) and the player
 * to move is drawn uniformly (maenv:523).  The table must stay allocated while it is set.  n_states = 0 (or a NULL
 * board pointer) switches back to setups.
 * start_index_d (optional, device, int32 [index_len]): start_index_d[global env id - index_env_base] receives the entry
 * every game was (re)started from -- maenv:524-527 maps the players through the entry's likely winner.  Global env id =
 * env_base + the env's position in the call, as everywhere else; ids outside [index_env_base, index_env_base +
 * index_len) are not recorded. */
int sx_config_set_start_states(sx_config *cfg, sx_state table, int64_t n_states, int32_t *start_index_d,
                               int64_t index_env_base, int64_t index_len);

/* Replaces penv.create_initial_state (penv:38 -> impl:213-249) + the setup samplers
 * (util:33-53 random, util:301-319 human).  Re-sets every env b with reset_mask_d[b] != 0 (all when
 * NULL).  Setups come from `setups_d` ([n_setups][setup_len] own-frame piece maps): rows
 * setup_idx_d[b][0..1] when given, else two Philox draws keyed by (seed, env_base + b, episode).
 * With SX_RESET_RANDOM_SHUFFLE in flags the table is ignored and pieces are shuffled on device. */
int sx_reset(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const uint8_t *reset_mask_d,
             const uint8_t *setups_d, int32_t n_setups, const int32_t *setup_idx_d, uint64_t seed, uint32_t flags,
             void *stream);

/* Bridge to the reference's dense state int64[34][R][C] (impl:16-60) -- `initial_state_override`
 * (maenv:551-553) and the facade methods use it.  status_d[b] != 0 marks a state the compact
 * layout cannot represent (never the case for states reached by play). */
int sx_import_ref_state(const sx_config *cfg, sx_state st, int64_t num_envs, const int64_t *dense_d,
                        const int8_t *player_d, uint8_t *status_d, void *stream);
int sx_export_ref_state(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t *dense_d, int8_t *player_d,
                        void *stream);

/* penv.get_state_from_player_perspective (penv:101 -> impl:646-675) on the device state: the dense state as
 * viewer_d[b] sees it (player -1: player layers swapped, board rotated 180 degrees; NULL = absolute frame).
 * This is what maenv puts in the observation dict under 'internal_state' (maenv:494-495). */
int sx_export_perspective_state(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *viewer_d,
                                int64_t *dense_d, void *stream);

/* impl:400-517 (spatial, in `player`'s frame) or impl:522-642 (1D, absolute frame): mask_d is
 * uint8 [num_envs][spatial_actions] or [num_envs][action_size].  player_d NULL = player to move. */
int sx_valid_mask(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *player_d, int32_t format,
                  uint8_t *mask_d, void *stream);

/* maenv:447-497 without the step: mask + normalised observations for player_d (NULL = to move). */
int sx_observe(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *player_d, sx_outputs out,
               void *stream);

/* impl:897-1045 (+ impl:835-849): applies actions_d[b] for the player to move; no rendering. */
int sx_step(const sx_config *cfg, sx_state st, int64_t num_envs, const int32_t *actions_d, int32_t action_format,
            uint32_t flags, sx_outputs out, void *stream);

/* The fused hot path, one launch per env-step: maenv.step (maenv:659-828) = action decode
 * (maenv:685-689) -> next state (impl:897) -> outcome (impl:835-849) -> [auto-reset] -> mask +
 * observations of the player to move (maenv:447-497) -> [uniform valid-action sample].
 * stats_d (optional, device, int64[8], accumulated with atomics): games finished, player +1 wins, player -1 wins,
 * invalid endings, rejected actions, actions processed, attacks, setup draws (re-draws of unplayable setups included). */
int sx_step_all(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const int32_t *actions_d,
                int32_t action_format, uint32_t flags, const uint8_t *setups_d, int32_t n_setups, uint64_t seed,
                sx_outputs out, int64_t *stats_d, void *stream);

/* Uniform draw over the valid entries of uint8 masks [num_envs][mask_len] (replaces maenv:830-834);
 * Philox4x32-10 keyed by (seed, env_base + b, step). */
int sx_sample_valid(const uint8_t *mask_d, int64_t num_envs, int32_t mask_len, int64_t env_base, uint64_t seed,
                    uint32_t step, int32_t *actions_d, void *stream);

/* Masked-logit action sampling, the step right upstream of sx_step_all in a rollout (replaces the CPU chooser
 * of examples/basic_game_loop.py:6-32 / README.md:38-65: softmax(logits + log(mask + 1e-8)) + np.random.choice).
 * Draws actions_d[b] ~ softmax(logits[b] / temperature) restricted to mask[b] != 0 (Gumbel-max, Philox4x32-10
 * keyed by (seed, env_base + b, step, entry)); invalid entries have probability exactly 0.  logits_d is
 * [num_envs][n_actions] of logits_dtype; logprob_d (optional) receives log p(action).  actions_d[b] = -1 when a
 * mask row has no valid entry.  A valid logit of -inf has probability 0; when every valid logit is -inf the action is
 * the lowest valid index and the log-probability NaN.  temperature must be > 0 with a finite reciprocal. */
int sx_sample_logits(const void *logits_d, int32_t logits_dtype, const uint8_t *mask_d, int64_t num_envs,
                     int32_t n_actions, int64_t env_base, uint64_t seed, uint32_t step, float temperature,
                     int32_t *actions_d, float *logprob_d, void *stream);

/* The same draw taken straight from the game STATE instead of a mask: the valid entries of the player to move are
 * regenerated from the compact state (~0.3 KB per game instead of the 3.7 KB mask row of a 10x10 board), then the
 * identical Gumbel-max runs over them -- same Philox key per (seed, env_base + b, step, entry), so for the same key it
 * returns the SAME action as sx_sample_logits on that state's mask.  logits_d is [num_envs][R*C*A] in the mover's
 * frame (what a policy fed with sx_step_all's observations emits).  A finished game or stuck player yields the noop
 * entry A-1 with log-probability 0 (impl:514-515). */
int sx_sample_policy(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const void *logits_d,
                     int32_t logits_dtype, uint64_t seed, uint32_t step, float temperature, int32_t *actions_d,
                     float *logprob_d, void *stream);

/* impl:854-891 (_get_heuristic_rewards_from_move): rewards_d[b] = reward_matrix[rank of the mover's piece on the
 * start square][rank of the opponent's piece on the end square, 0 = empty] for the action game b is about to play
 * (call it BEFORE the step).  reward_matrix_d is float32 [13][13] on the device; a no-op scores 0.  Like the
 * reference, the action is assumed to be valid. */
int sx_heuristic_rewards(const sx_config *cfg, sx_state st, int64_t num_envs, const int32_t *actions_d,
                         int32_t action_format, const float *reward_matrix_d, float *rewards_d, void *stream);

/* Determinization: n_samples complete game states per game that agree with what one player knows (for PIMC,
 * information-set MCTS, determinized rollouts, belief-model training).
 * The viewer of game b is viewer_d[b] (1 = player +1, anything else = player -1, as player_override of the step) or,
 * with viewer_d NULL, the player to move.  The HIDDEN cells of a game are the cells that hold a piece of the viewer's
 * opponent that is not CELL_REVEALED, on no obstacle; their HIDDEN MULTISET is the multiset of the true codes there (on
 * a reachable state: piece_amounts - captured - revealed alive, for the opponent: what the viewer can infer).
 * IMMOVABLE codes are FLAG (11) and BOMB (12).  S = hidden cells with CELL_STILL (never moved), I = immovable and
 * M = movable pieces of the hidden multiset.  A sample is a copy of the game in which the hidden multiset is placed on
 * the hidden cells uniformly at random among all placements that put no immovable piece on a cell without CELL_STILL.
 * Everything else stays byte for byte: aux, the capture list, every other cell byte, and the owner / revealed / still /
 * obstacle bits of the hidden cells; only their CELL_RANK nibble may differ.  A game without hidden cells is copied
 * unchanged; finished games are sampled like any other.  If I > S no placement exists (play never produces such a
 * state; sx_import_ref_state of a state in which a bomb or flag has moved can): the rows are copied unchanged and
 * status_d[b] = 1 (optional output; 0 otherwise).
 * Draws (exact, so a host reference can reproduce them): each hidden cell c (absolute index, < 256) of sample k of game
 * b gets one Philox4x32-10 block, key (seed lo, seed hi), counter (gid lo, gid hi, RNG_HIDDEN ^ draw, (k << 8) | c)
 * with gid = env_base + b and RNG_HIDDEN = 0x48494444; its words x and y are sort keys.  1. The still hidden cells are
 * ordered by (x, c) ascending; rank j < I receives the j-th immovable code in ascending order (flags before bombs).
 * 2. Every hidden cell not filled in step 1 is ordered by (y, c) ascending; rank j receives the j-th movable code in
 * ascending order.  Ranking by i.i.d. keys is a uniform permutation, so every consistent placement comes from exactly
 * one equally likely pair of (immovable, movable) placements; breaking key ties by the cell index biases this by less
 * than n^2 / 2^33 for n hidden cells.  Sample k of a game depends on (seed, draw, gid, k) only, not on n_samples, the
 * batch split or where env_base puts the game.
 * out has num_envs * n_samples rows (same strides as st); row b * n_samples + k is sample k of game b.  Refused:
 * n_samples < 1 or >= 2^24, a row count that overflows, out.board == st.board. */
int sx_sample_hidden_states(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base,
                            const int8_t *viewer_d, int32_t n_samples, uint64_t seed, uint32_t draw,
                            sx_state out, uint8_t *status_d, void *stream);

/* The children of a node, for search (PIMC, information-set MCTS, tree expansion).  The CHILDREN of game b are one per
 * legal move of its player to move: exactly the non-zero entries of sx_valid_mask(b) in the spatial format without the
 * noop channel A-1, each identified by its flat spatial index in that player's frame (what sx_step_all,
 * sx_sample_policy and a policy head use), in ascending index order.  A game with no legal move (a finished game, or an
 * imported state whose player to move is stuck) has zero children.  Nothing is random.
 * sx_count_moves: counts_d[b] (int32) = the number of children of game b.
 * sx_expand_moves: offsets_d is int64 [num_envs + 1], normally the exclusive prefix sum of the counts; child t of game b
 * is row offsets_d[b] + t of out (same strides as st), actions_d (int32) and the scalars of out_scalars.  The row holds,
 * byte for byte, what sx_step (SX_ACTION_SPATIAL, flags 0) makes of a copy of game b with action actions_d[row]: board
 * (padding included), aux, capture list, and reward, done, winner, ending_invalid, illegal (0, or 2 when the capture
 * list overflows) and player (any of them may be NULL).  st is never written.  offsets_d is not checked on the host: no
 * row outside [0, n_children) is written, a slot [offsets_d[b], offsets_d[b+1]) shorter than the count receives the
 * game's first children in order, and rows of a slot beyond the count are left untouched.  Refused: a null config,
 * state, out, actions_d or offsets_d, out.board == st.board, n_children < 0, and a non-null observation, mask,
 * next_action or terminal pointer in out_scalars.  num_envs <= 0 or n_children == 0: nothing to do. */
int sx_count_moves(const sx_config *cfg, sx_state st, int64_t num_envs, int32_t *counts_d, void *stream);
int sx_expand_moves(const sx_config *cfg, sx_state st, int64_t num_envs, const int64_t *offsets_d, int64_t n_children,
                    sx_state out, int32_t *actions_d, sx_outputs out_scalars, void *stream);

/* Random playouts, for scoring search leaves: every game of the batch is played on with uniformly random legal moves
 * until it ends or max_plies plies have been played, whichever comes first.  st is updated in place, like sx_step_all.
 * The move of each ply is the SX_SAMPLE_NEXT draw of sx_step_all for the state before that ply: Philox4x32-10 with key
 * (seed lo, seed hi) and counter (gid lo, gid hi, RNG_SAMPLE ^ (turn & 0xffff), episode), gid = env_base + b, first
 * output word w; the move is number __umulhi(w, n_moves) of the player to move's moves in ascending flat spatial index
 * (that player's frame).  So a playout of n plies equals, byte for byte (board with padding, aux, capture list and the
 * scalars below), this chain: a = that draw on the initial state; repeat { sx_step_all(a, SX_ACTION_SPATIAL,
 * SX_SAMPLE_NEXT, no auto-reset, same seed and env_base); a = next_action } until a step reports done or n steps have
 * run.  A playout therefore continues the chain a caller's last sx_step_all with that seed started (its first move is
 * the next_action that step returned), playout(a) then playout(b) equals playout(a + b), and the result depends on
 * (seed, gid, state) only, not on the batch split.  Two cases differ from that chain:
 *  - a game that is over at entry plays 0 plies and its rows are not written (a step of a finished game flips player);
 *  - a player to move with no legal move (only an imported state can be so) draws the noop entry A-1 and loses by it,
 *    as sx_step_all does with the 1D noop action (SX_ACTION_1D, action_size - 1); the spatial noop entry would be
 *    rejected as illegal, and the chain would never end.
 * Every game that is not over ends within max_turns - turn + 1 plies (turn limit), so max_plies = INT32_MAX plays every
 * game to its end.
 * Outputs per game, each optional (NULL): plies_d (int32) the plies played in this call; in out_scalars, as the step
 * that ended the game reported them (or, for a game over at entry, computed the same way from its aux): done (1 if the
 * game is over at the end of the call), winner, ending_invalid, reward; illegal (0, or 2 once the capture list has
 * overflowed: sticky, as in the step); player (to move at the end).  Refused: a null config or state tensor,
 * max_plies < 0, and a non-null observation, mask, next_action or terminal pointer in out_scalars.  num_envs <= 0:
 * nothing to do. */
int sx_playout(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, int32_t max_plies,
               uint64_t seed, int32_t *plies_d, sx_outputs out_scalars, void *stream);

/* Position keys, for transposition tables and information-set search: keys_d[b] (uint64) identifies game b.
 * SX_KEY_STATE: a key of the game as sx_export_ref_state exports it, the dense int64 [34][R][C] state plus the player to
 * move.  Two states with equal exports have equal keys; what the export does not hold has no effect (the aux episode
 * counter, board padding, the order of the capture-list entries, the overflow flag).  Two states whose exports differ
 * get different keys except with probability about 2^-64 per pair: among n distinct states some pair collides with
 * probability about n^2 / 2^65 (10^8 states: 3e-4).
 * SX_KEY_INFOSET: the state key of the same export after one change, for the viewer viewer_d[b] (1 = player +1,
 * anything else = player -1; NULL = the player to move, as sx_sample_hidden_states): on every HIDDEN cell of that call
 * (a piece of the viewer's opponent, code 1..12, not CELL_REVEALED, on no obstacle) the opponent's true-rank layer
 * (0 for player +1, 1 for player -1) holds the entry of its partially observable layer (3 / 4), UNKNOWN (13), instead
 * of the rank; and one more feature names the viewer.  So every state sx_sample_hidden_states draws for a viewer has
 * the information-set key of its source for that viewer, and a state's state key and its two information-set keys
 * differ by construction.
 * Construction (exact; no seed, no env_base, stable across calls and processes): Zobrist form, the XOR of
 * Z(c, l, x) over every non-zero dense entry x at (layer l, cell c) of layers 0-1 and 3-33 (layer 2, the obstacles, is
 * fixed by the configuration), plus Z(0, 34, player to move +1 / -1) and, for SX_KEY_INFOSET, Z(0, 35, viewer +1 / -1).
 * Z(c, l, x) = w0 | w1 << 32 with (w0, w1) the first two words of Philox4x32-10, key (0x53545241, 0x5445474f), counter
 * (c, l, (uint32_t)x, RNG_KEYS = 0x4b455953); c is the absolute cell index (the data layer: 0 turn, 1 over, 2 winner,
 * C max_turns, C + 1 invalid).  Captured counters enter as the dense counts: the compact capture list holds at most one
 * entry per (cell, owner, type), since a capture adds to an existing entry and sx_import_ref_state writes one entry per
 * non-zero counter.  XOR allows incremental updates (old word out, new word in).
 * Refused: a null config, state tensor or keys_d, an unknown mode, and a non-null viewer_d with SX_KEY_STATE.
 * num_envs <= 0: nothing to do. */
enum { SX_KEY_STATE = 0, SX_KEY_INFOSET = 1 };
int sx_state_keys(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *viewer_d, uint32_t mode,
                  uint64_t *keys_d, void *stream);

/* Monte Carlo tree search, a fixed number of iterations per root, every tree of the batch in one launch (one warp per
 * tree).  Game b is the root of its own tree of at most max_nodes nodes; node 0 is the root.  The nodes are stored
 * struct-of-arrays, each field int32 [num_envs, max_nodes] (node j of tree b at b * max_nodes + j):
 *   visits N; value W, the sum of the evaluations in absolute terms (+1: player +1 won); parent (-1 for the root);
 *   first_child (-1 while the node is not expanded); n_children; action, the flat spatial index of the move from the
 *   parent to the node in the frame of the parent's player to move (the sx_expand_moves / sx_step index; -1 for the root).
 * used (int32 [num_envs]) is the number of nodes allocated; entries at index used[b] and above are not written, and
 * neither is st.
 * Iteration i = 0 .. iterations - 1 of each tree:
 *  1. Descent: s = the root state, v = the root, path = [root].  Repeat: if s is over, stop.  If v has no children: let
 *     n be the number of legal moves of s's player to move; if n = 0 (a stuck player, only possible in an imported
 *     root) or used + n > max_nodes, stop (v stays a leaf); otherwise allocate n children at used .. used + n - 1, in
 *     ascending flat spatial index of their moves (the sx_expand_moves action list).  Choose a child c: the first child
 *     (lowest index) with N = 0 if there is one, else the argmax of the score below, ties to the lowest index.  Set s =
 *     the state after c's move (byte for byte what sx_step makes of s with that action), v = c, append c to the path;
 *     if c had N = 0 before this iteration, stop.
 *  2. Evaluation z in {-1, 0, +1}: if s is over, player +1's reward (the winner, 0 for a turn-limit ending); otherwise
 *     a random playout from s of at most max_plies plies, with sx_playout's rules (a stuck player plays the noop and
 *     loses) but the search's own draw: Philox4x32-10, key (seed lo, seed hi), counter (gid lo, gid hi,
 *     RNG_SEARCH ^ i, turn & 0xffff of the state before the ply), RNG_SEARCH = 0x54524545, gid = env_base + b, first
 *     output word w, move number __umulhi(w, n_moves) in ascending flat spatial index (sx_playout's numbering).  z is
 *     player +1's reward at the end of the playout, 0 if the ply cap cut it off.
 *  3. Backup: N += 1 and W += z on every node of the path.
 * Score of child c of node v, with sigma = +1 if player +1 is to move in v's state and -1 otherwise (PUCT with a uniform
 * prior), every operation float32, rounded to nearest, without FMA contraction:
 *   q = float(sigma * W_c) / float(N_c);  u = (c_explore * sqrt(float(N_v))) / float(1 + N_c);  score = q + u
 * with N_v and N_c the counts before this iteration's backup.  iterations <= 2^24 keeps every count and every |W| exact
 * in float32, so numpy float32 reproduces every score bit for bit.
 * Consequences: the tree depends only on (seed, gid, root state, iterations, max_nodes, max_plies, c_explore), not on the
 * batch split or the other games; the root has N = iterations; an expanded non-root node has N = 1 + the sum of its
 * children's N and an expanded root N = that sum; max_nodes = 1 makes the search `iterations` independent playouts of
 * the root; iterations = 0 gives used = 1.  One tree is one warp: a batch with fewer trees than the device's resident
 * warps leaves it partly idle.
 * Refused: a null config, state tensor or tree pointer, iterations < 0 or > 2^24, max_nodes < 1, max_plies < 0, and a
 * c_explore that is negative or not finite.  num_envs <= 0: nothing to do. */
typedef struct {
    int32_t *visits, *value, *parent, *first_child, *n_children, *action; /* [num_envs * max_nodes] */
    int32_t *used;                                                          /* [num_envs] */
} sx_tree;
int sx_search(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, int32_t iterations,
              int32_t max_nodes, int32_t max_plies, float c_explore, uint64_t seed, sx_tree tree, void *stream);

/* Guided tree search: PUCT selection and backup on the device, leaves evaluated by the caller (a policy prior and a
 * value from a network, AlphaZero style).  A simulation is three steps, none of which synchronises the host and all of
 * fixed shape (so they can run back to back or be captured in a CUDA graph):
 *   sx_guided_select (one launch) -> the caller's network on the leaf states -> sx_guided_backup (one launch).
 * Tree: game b is the root (node 0) of its own tree of at most max_nodes nodes, stored struct-of-arrays
 * [num_envs, max_nodes] (node j of tree b at b * max_nodes + j), with sx_tree's fields and two differences: value W is
 * float32, the sum of the values backed up in absolute terms (+1 = player +1 wins), and prior P (float32) is each
 * node's prior under its parent.  An empty tree is the root alone: used = 1, N = 0, W = 0, parent = -1,
 * first_child = -1, n_children = 0, action = -1, P = 1 in column 0; the caller writes it.  Columns at used[b] and above
 * hold anything.  A caller may rewrite the priors of existing nodes between calls (Dirichlet noise on the root's
 * children, say); nothing else in the tree is meant to be edited.
 * sx_guided_select reads the roots st and the tree and writes neither.  For every tree it descends from the root: at a
 * node v with children it takes the child c of highest score, ties to the lowest index, and steps into it (the state
 * sx_step makes of v's state with c's action); it stops at the first node without children or whose state is over.
 * Score, sigma = +1 if player +1 is to move at v and -1 otherwise, every operation float32, rounded to nearest, without
 * FMA contraction:
 *   q = N_c > 0 ? (sigma * W_c) / float(N_c) : fpu;  u = ((c_puct * P_c) * sqrt(float(N_v))) / float(1 + N_c);
 *   score = q + u
 * fpu is the value of an unvisited child from the mover's side.  Outputs per tree: leaf_states row b, the leaf's compact
 * state, byte for byte what the chain of steps along the path makes of the root (ready for sx_observe,
 * sx_valid_mask, sx_export_ref_state); leaf_node_d[b] (int32); leaf_kind_d[b] (int8, SX_LEAF_*): EVAL, the state is
 * not over and its player to move has a move; OVER; STUCK, the player to move has no move (only an imported root).
 * sx_guided_backup takes the leaves of the last select, logits_d [num_envs, R, C, A] (SX_DTYPE_F32 / BF16 / F16, the
 * layout of sx_sample_policy: the player to move's frame) and values_d (float32 [num_envs], from the side of the leaf's
 * player to move).  It needs no roots: the leaf's moves are regenerated from its leaf_states row.  For each tree:
 *  - expansion: an EVAL leaf without children gets, if used + n <= max_nodes, its n legal moves as children at
 *    used .. used + n - 1 in ascending flat spatial index (the sx_expand_moves list), with N = 0, W = 0,
 *    first_child = -1, n_children = 0, and P = the softmax of the logits over the legal entries only (expf, a float32
 *    sum, a correctly rounded division; a legal logit of -inf gets P = 0, and if every legal logit is -inf each child
 *    gets 1/n; NaN or +inf logits are undefined); used grows by n;
 *  - value z: EVAL sigma_leaf * values_d[b] (not clamped or checked); OVER player +1's reward (the winner, 0 for a
 *    turn-limit ending); STUCK -sigma_leaf (the stuck player loses, as in sx_search and sx_playout);
 *  - update: every node from the leaf to the root gets N += 1 and W += z (float32 add).
 * Consequences: the tree depends only on (root, the logits and values given, max_nodes, c_puct, fpu): no RNG, no
 * env_base, not the batch split; two selects without a backup between them return the same leaves; every expanded node,
 * the root included, has N = 1 + the sum of its children's N; after r rounds the root has N = r; a pool too small for
 * the next expansion stops the growth while values still back up.  The priors are the only transcendental result:
 * given them, every selection is reproduced bit for bit by numpy float32.
 * Refused: a null config, root state, tree field, leaf output, logits or values; leaf_states.board == st.board;
 * max_nodes < 1; a c_puct that is negative or not finite; an fpu that is not finite; an unknown logits dtype.
 * num_envs <= 0: nothing to do. */
enum { SX_LEAF_EVAL = 0, SX_LEAF_OVER = 1, SX_LEAF_STUCK = 2 };
typedef struct {
    int32_t *visits;                                          /* [num_envs * max_nodes] N */
    float *value;                                             /* W */
    int32_t *parent, *first_child, *n_children, *action;
    float *prior;                                             /* P */
    int32_t *used;                                            /* [num_envs] */
} sx_guided_tree;
int sx_guided_select(const sx_config *cfg, sx_state st, int64_t num_envs, sx_guided_tree tree, int32_t max_nodes,
                     float c_puct, float fpu, sx_state leaf_states, int32_t *leaf_node_d, int8_t *leaf_kind_d,
                     void *stream);
int sx_guided_backup(const sx_config *cfg, sx_state leaf_states, int64_t num_envs, sx_guided_tree tree,
                     int32_t max_nodes, const int32_t *leaf_node_d, const int8_t *leaf_kind_d, const void *logits_d,
                     int32_t logits_dtype, const float *values_d, void *stream);

/* Several leaves per tree in one round: L = leaves_per_tree leaves (1 <= L <= SX_GUIDED_MAX_LEAVES) under a virtual
 * loss, so that the caller's network evaluates num_envs * L leaves at once and S simulations take S / L rounds.  L is
 * chosen per call; different rounds may use different L.  num_envs counts trees; the leaf outputs have num_envs * L
 * rows, leaf j of tree b at row b * L + j.
 * sx_guided_select_many chooses the leaves of each tree in order j = 0 .. L-1, each a full descent from the root with
 * sx_guided_select's stopping rule.  Before leaf j is chosen, every node on the paths of leaves 0 .. j-1 (root and leaf
 * included) carries V = the number of those paths through it (all V are 0 for leaf 0), and the score of child c of v is
 *   n_c = N_c + V_c;  q = n_c > 0 ? (sigma * W_c - vl * float(V_c)) / float(n_c) : fpu;
 *   u = ((c_puct * P_c) * sqrt(float(N_v + V_v))) / float(1 + n_c);  score = q + u
 * float32, one rounding per operation, no contraction, ties to the lowest index.  vl = virtual_loss (finite,
 * 0 <= vl <= 2^24) is what each pending visit takes from the mover's value; vl = 0 is the "virtual visit" variant.
 * With V = 0, vl * 0 = +0 and sigma * W - (+0) = sigma * W (-0 included), so L = 1 gives sx_guided_select's leaves bit for
 * bit.  The pending visits live in inflight_d (int32 [num_envs * max_nodes], all zero before the call; it is all zero
 * again when the call's work is done; unused and may be null when L = 1).  The tree's fields are not written: two selects
 * without a backup return the same leaves.  Exactness needs N + V < 2^24 on every node.
 * sx_guided_backup_many takes those num_envs * L leaves, logits_d [num_envs * L, R, C, A] and values_d
 * [num_envs * L].  Per tree it processes the leaves in order j: an EVAL leaf whose node has no children at that point is
 * expanded with row j's logits if the pool has room after the expansions of leaves 0 .. j-1; then leaf j's z is added
 * along its path, as in sx_guided_backup.
 * Consequences: a node reached by several leaves of one round is expanded once, by the first of them, and every one of
 * them backs up its own value; the root gains N = L per round; every node has N = e + the sum of its children's N, e the
 * number of selections that ended at it; the tree depends only on (root, the logits and values given, max_nodes, c_puct,
 * fpu, vl, the L of each round), not on the batch split.  In the first round of an empty tree all L leaves are the root
 * (correct but wasteful: open with one L = 1 round).  L = 1 calls are sx_guided_select / sx_guided_backup exactly.
 * Refused: what sx_guided_select / sx_guided_backup refuse, L outside [1, SX_GUIDED_MAX_LEAVES], a virtual_loss that is
 * negative, not finite or above 2^24 (the bound keeps vl * V and sigma * W - vl * V finite), and a null inflight_d with
 * L > 1. */
enum { SX_GUIDED_MAX_LEAVES = 1024 };
int sx_guided_select_many(const sx_config *cfg, sx_state st, int64_t num_envs, sx_guided_tree tree, int32_t max_nodes,
                          float c_puct, float fpu, int32_t leaves_per_tree, float virtual_loss, int32_t *inflight_d,
                          sx_state leaf_states, int32_t *leaf_node_d, int8_t *leaf_kind_d, void *stream);
int sx_guided_backup_many(const sx_config *cfg, sx_state leaf_states, int64_t num_envs, sx_guided_tree tree,
                          int32_t max_nodes, int32_t leaves_per_tree, const int32_t *leaf_node_d,
                          const int8_t *leaf_kind_d, const void *logits_d, int32_t logits_dtype, const float *values_d,
                          void *stream);

/* Kernel/launch facts for the benchmark's roofline accounting. */
typedef struct {
    int32_t warps_per_block, blocks_per_sm, smem_bytes_per_block, num_sms, grid_blocks, regs_per_thread;
    int32_t background_bytes; /* shared-memory background images of a block (DESIGN.md "Rendering") */
    int32_t thread_per_game;  /* 1: the variant steps through sx_toy_kernel (one thread per game, boards of <= 16 cells) */
} sx_launch_info;
/* obs_mask bit 8: the launch shape used when the observation / mask outputs lie in compressible memory (sx_device_alloc) */
int sx_step_all_launch_info(const sx_config *cfg, uint32_t obs_mask /*1 po, 2 fo, 4 mask, 8 compressible*/, sx_launch_info *out);

/* ---- device memory ------------------------------------------------------------------------------
 * sx_device_alloc allocates `bytes` (0 counts as 1) of device memory on CUDA device `device`.  With
 * SX_ALLOC_COMPRESSIBLE it asks for memory with the generic data compression of the memory system
 * (cuMemCreate, CU_MEM_ALLOCATION_COMP_GENERIC): lines between L2 and DRAM are compressed, invisibly to kernels,
 * copy engines and torch, so an almost constant output image costs fewer DRAM bytes to write.  The size is rounded
 * up to the granularity of such memory (2 MB on B200).  When the device does not support it or the driver does
 * not grant it, the memory comes from cudaMalloc instead; *granted_flags (optional) tells which: SX_ALLOC_COMPRESSIBLE
 * or 0.  Any other flag bit is an error.  The contents are uninitialised.
 * sx_device_free releases such an allocation (NULL is a no-op; any other pointer is an error).  A compressible
 * allocation is unmapped only after the device has finished its work (cudaDeviceSynchronize), as cudaFree would.
 * sx_device_alloc_info reports an allocation's requested size and granted flags and, optionally, how many
 * allocations of the library are live (ptr may be NULL for the count alone). */
#define SX_ALLOC_COMPRESSIBLE 1u
int sx_device_alloc(int32_t device, uint64_t bytes, uint32_t flags, void **ptr, uint32_t *granted_flags);
int sx_device_free(void *ptr);
int sx_device_alloc_info(const void *ptr, uint64_t *bytes, uint32_t *granted_flags, int64_t *live_allocations);

/* ---- host-buffer convenience object (the e2e path: host actions in, host tensors out) ------------
 * Owns device state + output buffers for num_envs games on the current device (the observation and mask buffers
 * compressible where the device grants it, see sx_device_alloc) and pipelines
 * H2D(actions) -> sx_step_all -> D2H(outputs) in chunks over internal streams. */
typedef struct sx_host_env sx_host_env;
int sx_host_env_create(const sx_config *cfg, int64_t num_envs, int64_t env_base, uint32_t obs_mask, uint32_t flags,
                       const uint8_t *setups_host, int32_t n_setups, uint64_t seed, int32_t n_chunks,
                       sx_host_env **out);
void sx_host_env_destroy(sx_host_env *env);
/* host pointers; pinned memory recommended.  reset fills the outputs for the first player. */
int sx_host_env_reset(sx_host_env *env, sx_outputs host_out);
int sx_host_env_step(sx_host_env *env, const int32_t *actions_host, sx_outputs host_out);
/* same with an explicit action format (SX_ACTION_1D for maenv.step(..., is_spatial_index=False)) and per-call
 * flags (e.g. SX_ALLOW_OSCILLATION) instead of the ones given at creation */
int sx_host_env_step_ex(sx_host_env *env, const int32_t *actions_host, int32_t action_format, uint32_t flags,
                        sx_outputs host_out);
/* device-resident variant used for the kernel-only measurement: no host copies */
int sx_host_env_step_device(sx_host_env *env, int32_t use_sampled_actions);
int sx_host_env_sync(sx_host_env *env);
/* device pointers of the object's state (for sx_import_ref_state / sx_export_ref_state / sx_observe on it, e.g.
 * maenv's initial_state_override) and, optionally, of its device-side output buffers */
int sx_host_env_state(sx_host_env *env, sx_state *state_out, sx_outputs *device_outputs_out);

#ifdef __cplusplus
}
#endif
#endif /* STRATEGO_B200_H */
