"""``BatchedStrategoEnv``: the batched, device-resident variant of ``StrategoMultiAgentEnv``.

``num_envs`` independent games live on one GPU in the compact struct-of-arrays layout; ``step`` is ONE
launch of the fused sm_100a kernel (action decode -> move / combat -> outcome -> auto-reset -> next
player's mask + observations [-> uniform valid-action sample]) and everything it returns is a torch CUDA
tensor -- nothing crosses PCIe unless the caller asks.  Observation keys and layouts are the reference's
(``ObservationComponents``; HWC float32 observations, or bfloat16 / float16 with ``obs_dtype``; the mask is uint8
instead of the reference's int64).

Semantics that differ from the one-game API because many games advance at once:
  * obs / mask / ``player`` are always for the player to move next in each game, in that player's frame;
  * when a game ends during ``step`` the returned ``done`` / ``winner`` / ``game_result_was_invalid`` / rewards
    describe the finished game, and (with ``auto_reset=True``) the observation is already the first
    observation of the next game.  The terminal observations the reference hands to BOTH players (maenv:772-773)
    arrive in ``infos['terminal_observation']`` when the env is built with ``terminal_observations=True``
    (rows of games with ``done``; written by the same kernel launch, before the re-set);
  * ``same_start_pos_everytime`` (maenv:352-354) fixes ONE setup per env (the reference has one env), ``repeat_games_
    from_other_side`` (maenv:530-534) replays every env's previous initial position from the other side on its odd
    episodes, ``random_player_assignment`` (maenv:537-543) draws a +-1 agent map per env and game: ``player``, the
    reward dict and ``infos['winner']`` are then expressed in agent ids, ``infos['player_map']`` holds the map;
  * an illegal action leaves that game untouched and sets ``illegal_action`` (the reference raises
    ``ValueError``, impl:899-902); pass ``raise_on_illegal=True`` to get the exception (costs a host sync).
"""
from typing import Optional

import numpy as np
import torch

from . import sharding
from .config import HUMAN_INIT_TABLE, VERSION_CONFIGS, as_version
from .engine import DeviceState, Expansion, Leaves, SearchTree, StrategoEngine, load_setup_table, obs_dtype_code
from .enums import GameVersions, ObservationComponents, ObservationModes
from .stratego_multiagent_env import DEFAULT_CONFIG, with_base_config

OC = ObservationComponents


class BatchedStrategoEnv:
    def __init__(self, env_config=None, num_envs: int = 1024, device=None, seed: int = 0, env_base: int = 0,
                 auto_reset: bool = True, sample_actions: bool = False, raise_on_illegal: bool = False,
                 terminal_observations: bool = False, obs_dtype=torch.float32):
        """obs_dtype: element type of the observations (torch.float32, torch.bfloat16 or torch.float16; StrategoEngine)"""
        obs_dtype_code(obs_dtype)  # a bad dtype is a ValueError before anything needs a device
        cfg = with_base_config(DEFAULT_CONFIG, env_config if env_config else {})
        cfg['version'] = as_version(cfg['version'])
        self.version = cfg['version']
        version_config = VERSION_CONFIGS[self.version]
        cfg = with_base_config(version_config, cfg)
        for key in ('vs_human', 'vs_bot'):
            if cfg[key]:
                raise NotImplementedError("%s is a single-game option (use StrategoMultiAgentEnv)" % key)
        assert not (cfg['human_inits'] and cfg['curriculum_start_states_path'])  # maenv:332
        self.use_curriculum_inits = bool(cfg['curriculum_start_states_path'])
        self.same_start_pos_everytime = bool(cfg['same_start_pos_everytime'])
        self.repeat_games_from_other_side = bool(cfg['repeat_games_from_other_side'])
        self.random_player_assignment = bool(cfg['random_player_assignment'])
        assert not (self.random_player_assignment and self.repeat_games_from_other_side)  # maenv:358
        assert not (self.use_curriculum_inits and (self.random_player_assignment or self.repeat_games_from_other_side))
        self.terminal_observations = bool(terminal_observations)
        mode = cfg['observation_mode']
        mode = mode if isinstance(mode, ObservationModes) else ObservationModes(mode)
        self.observation_mode = mode
        self._po = mode in (ObservationModes.PARTIALLY_OBSERVABLE, ObservationModes.BOTH_OBSERVATIONS)
        self._fo = mode in (ObservationModes.FULLY_OBSERVABLE, ObservationModes.BOTH_OBSERVATIONS)
        self.penalize_ties = bool(cfg['penalize_ties'])
        self.include_internal_state = bool(cfg['observation_includes_internal_state'])
        self.human_inits = bool(cfg['human_inits'])
        if self.human_inits and self.version not in HUMAN_INIT_TABLE:
            raise ValueError("Human inits not supported with {} game version".format(self.version.value))

        self.num_envs, self.seed, self.env_base = int(num_envs), int(seed), int(env_base)
        self.auto_reset, self.sample_actions, self.raise_on_illegal = auto_reset, sample_actions, raise_on_illegal
        self.engine = StrategoEngine({k: cfg[k] for k in version_config}, device=device,
                                     p2_rot180=not self.human_inits, obs_channel_mode=cfg['obs_channel_mode'],
                                     obs_dtype=obs_dtype)
        self.device = self.engine.device
        self.rows, self.columns = self.engine.rows, self.engine.columns
        self.spatial_action_size = self.engine.spatial_action_size
        self.setups = (self.engine.upload_setups(load_setup_table(HUMAN_INIT_TABLE[self.version]))
                       if self.human_inits else None)
        self.state: DeviceState = self.engine.alloc_state(self.num_envs)
        self.out = self.engine.alloc_outputs(self.num_envs, partial=self._po, full=self._fo, mask=True,
                                             sample=sample_actions, terminal=self.terminal_observations)
        # random_player_assignment: agent id of internal player +1, per env and game (maenv:537-543)
        self.player_map = torch.ones(self.num_envs, dtype=torch.int8, device=self.device)
        self._map_rng = torch.Generator(device=self.device)
        self._map_rng.manual_seed((self.seed * 1000003 + self.env_base) & (2 ** 62 - 1))
        self.stats = torch.zeros(8, dtype=torch.int64, device=self.device)
        # curriculum starts (maenv:341-351, 519-527): every game starts from a drawn entry of the file's states, the player
        # to move is drawn, and agent +1 is the entry's likely winner ("player 1 gets the advantage", maenv:525-527)
        self._start_index = self._likely_winner = None
        if self.use_curriculum_inits:
            from . import setups as _setups
            states, winners = _setups.load_curriculum_table(cfg['curriculum_start_states_path'])
            self._likely_winner = torch.as_tensor(np.asarray(winners), dtype=torch.int8, device=self.device)
            self._start_index = self.engine.set_start_states(torch.as_tensor(np.asarray(states)), self.num_envs,
                                                             self.env_base)
        self._spare_actions = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device) if sample_actions else None

    @classmethod
    def from_distributed(cls, env_config=None, envs_per_rank: Optional[int] = None, global_envs: Optional[int] = None,
                         **kwargs) -> "BatchedStrategoEnv":
        """one process per GPU (torchrun): this rank's shard of the global batch on cuda:LOCAL_RANK"""
        shard = sharding.current_shard(global_envs=global_envs, envs_per_rank=envs_per_rank)
        env = cls(env_config, num_envs=shard.num_local, device=torch.device("cuda", shard.local_rank),
                  env_base=shard.env_base, **kwargs)
        env.shard = shard
        return env

    # ---- observation dict ---------------------------------------------------------------------------
    def _draw_player_map(self, where: Optional[torch.Tensor] = None):
        """np.random.random() < 0.5 -> identity, else swapped (maenv:538-543), per env; `where` selects the envs whose
        game just (re)started"""
        new = torch.where(torch.rand(self.num_envs, generator=self._map_rng, device=self.device) < 0.5, 1, -1).to(torch.int8)
        self.player_map = new if where is None else torch.where(where, new, self.player_map)

    def _obs(self) -> dict:
        player = self.out["player"] * self.player_map if self._mapped else self.out["player"]
        d = {OC.VALID_ACTIONS_MASK.value: self.out["valid_mask"], "player": player}
        if self._po:
            d[OC.PARTIAL_OBSERVATION.value] = self.out["partial_obs"]
        if self._fo:
            d[OC.FULL_OBSERVATION.value] = self.out["full_obs"]
        if self.include_internal_state:
            d[OC.INTERNAL_STATE.value] = self.engine.export_perspective_state(self.state, self.out["player"])
        if self.sample_actions:
            d["sampled_action"] = self.out["next_action"]
        return d

    @property
    def _mapped(self) -> bool:
        """agent ids differ from internal player ids: random_player_assignment (maenv:537-543) or curriculum (maenv:524-527)"""
        return self.random_player_assignment or self.use_curriculum_inits

    def _curriculum_player_map(self):
        """maenv:526: player_map(p) = p * likely_winner of the entry the env's current game was started from"""
        self.player_map = self._likely_winner[self._start_index.long()]

    def reset(self, reset_mask: Optional[torch.Tensor] = None) -> dict:
        """(re)starts every game (or those with reset_mask[b] != 0) from freshly sampled setups"""
        self.engine.reset(self.state, seed=self.seed, env_base=self.env_base, reset_mask=reset_mask,
                          setups=self.setups, shuffle=self.setups is None, same_setup=self.same_start_pos_everytime,
                          repeat_other_side=self.repeat_games_from_other_side)
        if self.random_player_assignment:
            self._draw_player_map(None if reset_mask is None else reset_mask != 0)
        if self.use_curriculum_inits:
            self._curriculum_player_map()
        self.engine.observe(self.state, out=self.out, partial=self._po, full=self._fo, mask=True)
        if self.sample_actions:
            self.out["next_action"] = self.engine.sample_valid(self.out["valid_mask"], seed=self.seed, step=0,
                                                               env_base=self.env_base)
        return self._obs()

    def step(self, actions: torch.Tensor):
        """actions: int32 [num_envs], flat index into (R, C, A) in the mover's frame (what maenv.step takes)."""
        if actions.dtype != torch.int32:
            actions = actions.to(torch.int32)
        actions = actions.contiguous()
        if self.sample_actions and actions.data_ptr() == self.out["next_action"].data_ptr():
            # the caller plays the sampled actions: ping-pong so the kernel does not overwrite its own input
            self.out["next_action"], self._spare_actions = self._spare_actions, self.out["next_action"]
        self.engine.step_all(self.state, actions, self.out, env_base=self.env_base, auto_reset=self.auto_reset,
                             sample_next=self.sample_actions, setups=self.setups, shuffle=self.setups is None,
                             seed=self.seed, stats=self.stats, same_setup=self.same_start_pos_everytime,
                             repeat_other_side=self.repeat_games_from_other_side)
        out = self.out
        if self.raise_on_illegal and bool(out["illegal"].any().item()):
            bad = torch.nonzero(out["illegal"]).flatten().tolist()[:8]
            raise ValueError("Couldn't get the next state because the move wasn't valid. (envs %s)" % bad)
        reward_p1 = out["reward"]
        if self.penalize_ties:  # maenv:803-805: both players get -0.5 for a tie
            tie = (out["done"] != 0) & (out["winner"] == 0)
            reward_p1 = torch.where(tie, torch.full_like(reward_p1, -0.5), reward_p1)
            reward_p2 = torch.where(tie, torch.full_like(reward_p1, -0.5), -out["reward"])
        else:
            reward_p2 = -out["reward"]
        rewards = {1: reward_p1, -1: reward_p2}
        dones = out["done"]
        infos = {"winner": out["winner"], "game_result_was_invalid": out["ending_invalid"],
                 "illegal_action": out["illegal"]}
        if self._mapped:  # maenv:807-811: everything keyed by player is re-keyed by agent id
            m = self.player_map
            rewards = {1: torch.where(m == 1, reward_p1, reward_p2), -1: torch.where(m == 1, reward_p2, reward_p1)}
            infos["winner"] = out["winner"] * m
            infos["player_map"] = m
        if self.terminal_observations:
            # index 0 / 1 of the side buffers = player +1 / -1 (or agent +1 / -1 under random_player_assignment)
            term = {}
            for key, name in ((OC.PARTIAL_OBSERVATION.value, "terminal_partial_obs"), (OC.FULL_OBSERVATION.value, "terminal_full_obs")):
                if name in out:
                    t = out[name]
                    if self._mapped:
                        swap = (self.player_map == -1).view(-1, 1, 1, 1, 1)
                        t = torch.where(swap, t.flip(1), t)
                    term[key] = t
            infos["terminal_observation"] = {1: {k: v[:, 0] for k, v in term.items()}, -1: {k: v[:, 1] for k, v in term.items()}}
        obs = self._obs()
        if self.use_curriculum_inits and self.auto_reset:
            self._curriculum_player_map()  # the kernel re-started the finished games from freshly drawn entries
            obs["player"] = self.out["player"] * self.player_map
        if self.random_player_assignment and self.auto_reset:
            # games that ended were re-set inside the kernel and the returned observation already belongs to their NEXT
            # game: that game gets a fresh agent map (maenv:537-543), and its `player` is expressed in it
            self._draw_player_map(dones != 0)
            obs["player"] = self.out["player"] * self.player_map
        return obs, rewards, dones, infos

    def sample_actions_from_logits(self, logits: torch.Tensor, temperature: float = 1.0, return_logprob: bool = False):
        """masked-logit sampling for the current observation's mask (one kernel; the policy's logits stay on the
        GPU).  logits: [num_envs, R*C*A] or [num_envs, R, C, A], float32 / bfloat16 / float16."""
        self._policy_step = getattr(self, "_policy_step", 0) + 1
        # drawn from the compact state (sx_sample_policy): the mask the step kernel just wrote is not read back
        return self.engine.sample_policy(self.state, logits, seed=self.seed, step=self._policy_step,
                                         env_base=self.env_base, temperature=temperature,
                                         return_logprob=return_logprob)

    def heuristic_rewards(self, actions: torch.Tensor, reward_matrix: torch.Tensor) -> torch.Tensor:
        """impl:854-891 for the whole batch: reward_matrix[mover's rank, captured rank] (float32 [13, 13]) of the action
        each game is about to play -- call it before ``step(actions)``"""
        if actions.dtype != torch.int32:
            actions = actions.to(torch.int32)
        return self.engine.heuristic_rewards(self.state, actions.contiguous(), reward_matrix)

    def observe(self, player: Optional[torch.Tensor] = None, partial=True, full=True, mask=True) -> dict:
        """mask + observations for an arbitrary viewer per game (+1 / -1; default: the player to move)"""
        o = self.engine.observe(self.state, player, partial=partial, full=full, mask=mask)
        d = {"player": o["player"]}
        if mask:
            d[OC.VALID_ACTIONS_MASK.value] = o["valid_mask"]
        if partial:
            d[OC.PARTIAL_OBSERVATION.value] = o["partial_obs"]
        if full:
            d[OC.FULL_OBSERVATION.value] = o["full_obs"]
        return d

    def sample_hidden_states(self, n_samples: int = 1, viewer: Optional[torch.Tensor] = None) -> DeviceState:
        """Determinized copies of the current games (StrategoEngine.sample_hidden_states): ``n_samples`` states per game
        in which the pieces the viewer has not seen are re-placed uniformly at random, consistently with what the viewer
        knows.  viewer: None (the player to move) or an integer tensor [num_envs] of INTERNAL player ids (+1 / -1), the
        ids ``observe`` takes -- not the agent ids of ``random_player_assignment`` or curriculum starts.  Uses the env's
        seed and env_base and a draw counter that advances per call, so repeated calls give fresh samples.  Returns a
        DeviceState of num_envs * n_samples rows (row b * n_samples + k = sample k of game b) for ``self.engine``."""
        self._hidden_draw = getattr(self, "_hidden_draw", 0) + 1
        return self.engine.sample_hidden_states(self.state, n_samples=n_samples, viewer=viewer, seed=self.seed,
                                                draw=self._hidden_draw, env_base=self.env_base)

    def expand_moves(self) -> Expansion:
        """The children of the current games (StrategoEngine.expand_moves): one per legal move of the player to move, in
        ascending flat spatial index, each with the state and step outputs that move leads to.  Player ids in the result
        (``player``) are INTERNAL (+1 / -1), as for ``sample_hidden_states``.  One host synchronisation per call."""
        return self.engine.expand_moves(self.state)

    def search(self, iterations: int, seed: int = 0, max_nodes: Optional[int] = None, max_plies: Optional[int] = None,
               c_explore: float = 1.0):
        """Monte Carlo tree search from every current game (StrategoEngine.search), with this env's env_base: a
        SearchTree with one tree per env.  Player ids in it (``root_player``, values in absolute terms) are INTERNAL
        (+1 / -1).  The games are not changed.  No host synchronisation."""
        return self.engine.search(self.state, iterations, max_nodes=max_nodes, max_plies=max_plies, c_explore=c_explore,
                                  seed=seed, env_base=self.env_base)

    def guided_tree(self, max_nodes: int) -> SearchTree:
        """An empty guided tree per current game (StrategoEngine.guided_tree)."""
        return self.engine.guided_tree(self.state, max_nodes)

    def guided_select(self, tree: SearchTree, c_puct: float = 1.25, fpu: float = 0.0, leaves_per_tree: int = 1,
                      virtual_loss: float = 1.0) -> Leaves:
        """``leaves_per_tree`` leaves per tree rooted at the current games (StrategoEngine.guided_select); back the
        evaluated leaves up with ``self.engine.guided_backup``, which needs no roots."""
        return self.engine.guided_select(self.state, tree, c_puct=c_puct, fpu=fpu, leaves_per_tree=leaves_per_tree,
                                         virtual_loss=virtual_loss)

    def state_keys(self, info_set: bool = False, viewer: Optional[torch.Tensor] = None) -> torch.Tensor:
        """64-bit keys of the current games (StrategoEngine.state_keys), int64 [num_envs]: of the position, or with
        info_set=True of what the viewer knows.  viewer: None (the player to move) or an integer tensor [num_envs] of
        INTERNAL player ids (+1 / -1), as for ``sample_hidden_states``."""
        return self.engine.state_keys(self.state, info_set=info_set, viewer=viewer)

    # ---- checkpoint / interop in the reference's dense layout ---------------------------------------------
    def export_states(self):
        """(int64 [B, 34, R, C], int8 [B] player to move) -- the reference's state layout (impl:16-60)"""
        return self.engine.export_ref_state(self.state)

    def import_states(self, dense: torch.Tensor, player: Optional[torch.Tensor] = None):
        self.engine.import_ref_state(dense, player, state=self.state)

    def reduce_stats(self) -> dict:
        """end-of-run statistics summed over all ranks (the only collective this package issues)"""
        return sharding.stats_dict(sharding.reduce_stats(self.stats.clone()))
