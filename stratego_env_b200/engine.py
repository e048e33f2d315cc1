"""Torch-facing wrapper of the C ABI (include/stratego_b200.h).

``StrategoEngine`` owns one ``sx_config`` (a game variant) and exposes the kernels on torch CUDA
tensors: torch is used only for device memory and streams; every operation below is one launch of
the hand-written sm_100a kernels in ``csrc/`` on the current CUDA stream.
"""
import ctypes as C
import os
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import _lib
from .config import (captured_lut, obstacle_map, original_captured_lut, original_po_rank_lut, original_rank_lut,
                     original_unit_lut, piece_amounts_array, recent_moves_lut, unit_channel_lut)
from .enums import NUM_STATE_LAYERS

DATA_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")


def load_setup_table(name: str) -> np.ndarray:
    """uint8 [n, 40] human setups ('barrage' or 'standard'), baked by tools/gen_setup_tables.py from the
    reference's inits/*.py through its own transform (util:241-275)."""
    with np.load(os.path.join(DATA_DIR, "%s_setups.npz" % name)) as d:
        return np.ascontiguousarray(d["setups"], dtype=np.uint8)


@dataclass
class DeviceState:
    """Compact struct-of-arrays game state (DESIGN.md "State layout")."""
    board: torch.Tensor     # uint8  [B, board_stride]
    aux: torch.Tensor       # int16  [B, 8]
    captured: torch.Tensor  # uint16-as-int16 [B, captured_stride]

    @property
    def num_envs(self) -> int:
        return self.board.shape[0]

    def as_struct(self) -> _lib.SxState:
        return _lib.SxState(self.board.data_ptr(), self.aux.data_ptr(), self.captured.data_ptr())

    def clone(self) -> "DeviceState":
        return DeviceState(self.board.clone(), self.aux.clone(), self.captured.clone())

    def select(self, lo: int, hi: int) -> "DeviceState":
        return DeviceState(self.board[lo:hi], self.aux[lo:hi], self.captured[lo:hi])


@dataclass
class Expansion:
    """The children of a batch of games (StrategoEngine.expand_moves), T rows in all; game b's children are rows
    offsets[b] .. offsets[b + 1] - 1 of every field."""
    states: DeviceState           # T children, in the engine's strides
    actions: torch.Tensor         # int32 [T] flat spatial index of the move, in the parent's player-to-move frame
    parent: torch.Tensor          # int64 [T] game each child comes from
    offsets: torch.Tensor         # int64 [B + 1] exclusive prefix sum of the number of children per game
    reward: torch.Tensor          # float32 [T] as step returns them for that move
    done: torch.Tensor            # uint8 [T]
    winner: torch.Tensor          # int8 [T]
    ending_invalid: torch.Tensor  # uint8 [T]
    illegal: torch.Tensor         # uint8 [T] 0, or 2 when the capture list overflowed
    player: torch.Tensor          # int8 [T] player to move in the child (+1 / -1)


@dataclass
class Playout:
    """What StrategoEngine.playout reports per game of the batch (B rows each)."""
    plies: torch.Tensor           # int32 [B] plies played in this call
    reward: torch.Tensor          # float32 [B] player +1's reward if the game is over at the end, else 0
    done: torch.Tensor            # uint8 [B] the game is over at the end of the call
    winner: torch.Tensor          # int8 [B] +1 / -1, 0 for a draw by the turn limit or a game still running
    ending_invalid: torch.Tensor  # uint8 [B] the game ended by the turn limit
    illegal: torch.Tensor         # uint8 [B] 0, or 2 once the capture list has overflowed
    player: torch.Tensor          # int8 [B] player to move at the end (+1 / -1)


@dataclass
class SearchTree:
    """The trees StrategoEngine.search builds, one per game of the batch (sx_search), or the trees of a guided search
    (StrategoEngine.guided_tree / guided_select / guided_backup).  Node j of tree b is column j of the [B, max_nodes]
    fields; node 0 is the root.  Columns at used[b] and above are not written (they hold anything)."""
    visits: torch.Tensor       # int32 [B, max_nodes] N
    value: torch.Tensor        # int32 (search) / float32 (guided) [B, max_nodes] W: sum of the values, +1 = player +1 won
    parent: torch.Tensor       # int32 [B, max_nodes] -1 for the root
    first_child: torch.Tensor  # int32 [B, max_nodes] -1 while the node is not expanded
    n_children: torch.Tensor   # int32 [B, max_nodes]
    action: torch.Tensor       # int32 [B, max_nodes] flat spatial index of the move from the parent (its player's frame)
    used: torch.Tensor         # int32 [B] nodes allocated
    root_player: torch.Tensor  # int8 [B] player to move at the root (+1 / -1)
    mask_shape: tuple          # (R, C, A): the spatial valid-mask shape of one game
    prior: Optional[torch.Tensor] = None  # float32 [B, max_nodes] P, the prior under the parent (guided trees only)
    # int32 [B, max_nodes], all zero between calls: the pending visits of a round with several leaves per tree
    # (guided_select with leaves_per_tree > 1 creates it the first time; None until then)
    inflight: Optional[torch.Tensor] = None

    def root_stats(self):
        """(visits, values) of the root's children, shaped like the valid mask [B, R, C, A]: visits int32, values in the
        dtype of ``value``.  At the entry of each legal move of the root's player to move, its child's N and W, the value
        seen from the root's player to move (+1 = that player won); zero elsewhere, and everywhere for a root that was
        never expanded.  Torch ops only (a scatter over the nodes whose parent is the root), no host synchronisation."""
        B, M = self.visits.shape
        n = int(np.prod(self.mask_shape))
        live = (self.parent == 0) & (torch.arange(M, device=self.visits.device)[None, :] < self.used[:, None].long())
        idx = torch.where(live, self.action.long(), 0)
        zero = torch.zeros((), dtype=torch.int32, device=self.visits.device)
        vzero = torch.zeros((), dtype=self.value.dtype, device=self.visits.device)
        sign = self.root_player.to(self.value.dtype)[:, None]
        visits = torch.zeros(B, n, dtype=torch.int32, device=self.visits.device)
        values = torch.zeros(B, n, dtype=self.value.dtype, device=self.visits.device)
        visits.scatter_add_(1, idx, torch.where(live, self.visits, zero))
        values.scatter_add_(1, idx, torch.where(live, self.value * sign, vzero))
        return visits.view(B, *self.mask_shape), values.view(B, *self.mask_shape)


@dataclass
class Leaves:
    """The leaves StrategoEngine.guided_select picked, per_tree per tree (B * per_tree rows each; leaf j of tree b is
    row b * per_tree + j)."""
    states: DeviceState        # the leaf's state: byte for byte what the steps along its path make of the root
    node: torch.Tensor         # int32 [B * per_tree] the leaf's node index in its tree
    kind: torch.Tensor         # int8 [B * per_tree] LEAF_EVAL (to be evaluated), LEAF_OVER (game over) or LEAF_STUCK
    per_tree: int = 1          # leaves per tree (leaves_per_tree of the select)


LEAF_EVAL, LEAF_OVER, LEAF_STUCK = _lib.SX_LEAF_EVAL, _lib.SX_LEAF_OVER, _lib.SX_LEAF_STUCK

# observation element types (sx_config_desc::obs_dtype)
OBS_DTYPES = {torch.float32: _lib.SX_DTYPE_F32, torch.bfloat16: _lib.SX_DTYPE_BF16, torch.float16: _lib.SX_DTYPE_F16}


def obs_dtype_code(obs_dtype) -> int:
    """the sx_config_desc::obs_dtype value of a torch dtype; ValueError for anything but float32 / bfloat16 / float16"""
    code = OBS_DTYPES.get(obs_dtype) if isinstance(obs_dtype, torch.dtype) else None
    if code is None:
        raise ValueError("obs_dtype must be torch.float32, torch.bfloat16 or torch.float16, not %r" % (obs_dtype,))
    return code


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


class DeviceAllocation:
    """One device allocation of the library (sx_device_alloc): ``nbytes`` bytes on ``device``, compressible
    (``compressed``) when asked for and granted.  It exposes itself as a uint8 [nbytes] array through
    ``__cuda_array_interface__``; tensors made from it with ``torch.as_tensor`` hold a reference to it, so the memory is
    freed (sx_device_free) once, when the last of them is gone."""

    def __init__(self, device, nbytes: int, compressible: bool = True):
        lib = _lib.load()
        ptr, granted = C.c_void_p(), C.c_uint32()
        device = torch.device(device)
        index = device.index if device.index is not None else torch.cuda.current_device()
        _lib.check(lib.sx_device_alloc(index, int(nbytes), _lib.SX_ALLOC_COMPRESSIBLE if compressible else 0,
                                       C.byref(ptr), C.byref(granted)), "sx_device_alloc")
        self._lib, self.ptr, self.nbytes = lib, ptr.value, int(nbytes)
        self.compressed = bool(granted.value & _lib.SX_ALLOC_COMPRESSIBLE)
        self.__cuda_array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False),
                                         "strides": None, "version": 3}

    def __del__(self):
        ptr, self.ptr = getattr(self, "ptr", None), None
        if ptr:
            self._lib.sx_device_free(ptr)


class StrategoEngine:
    def __init__(self, game_version_config: dict, device=None, p2_rot180: bool = True, normalize: bool = True,
                 capture_capacity: int = 0, obs_channel_mode: str = 'extended', obs_dtype=torch.float32,
                 compressible_outputs: Optional[bool] = None):
        """normalize=False: observations carry the raw channel values of the procedural layer (penv:157-173)
        instead of the env-level [-1, 1] normalisation (maenv:499-508).  obs_channel_mode='original' selects the
        deprecated 32 / 33-channel observations (maenv:370-375, impl:1048-1197).  obs_dtype: element type of every
        observation output, torch.float32, torch.bfloat16 or torch.float16; a 16-bit observation equals the float32 one
        cast with ``.to(obs_dtype)`` (round to nearest even), at half the bytes written.
        compressible_outputs: where ``alloc_outputs`` puts the observation and mask planes.  None (default): in one
        allocation of the library with the device's generic data compression when the device grants it (the planes are
        an almost constant image, so the DRAM write stream that bounds the fused kernel shrinks; results are the same
        bytes), plain device memory otherwise; True: the same, but an error when compression is not granted; False:
        ``torch.empty`` as before.  ``outputs_compressed`` tells what the last ``alloc_outputs`` got."""
        if obs_channel_mode not in ('extended', 'original'):
            raise ValueError("obs_channel_mode must be 'extended' or 'original'")
        if compressible_outputs is not None and not isinstance(compressible_outputs, bool):
            raise ValueError("compressible_outputs must be None, True or False, not %r" % (compressible_outputs,))
        self.compressible_outputs = compressible_outputs
        self.outputs_compressed = False
        desc_obs_dtype = obs_dtype_code(obs_dtype)
        self.obs_dtype = obs_dtype
        self.obs_channel_mode = obs_channel_mode
        original = obs_channel_mode == 'original'
        if not torch.cuda.is_available():
            raise _lib.StrategoB200Error("StrategoEngine needs a CUDA device; there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else "cuda")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.game_version_config = game_version_config
        cfg = game_version_config
        self.rows, self.columns = int(cfg['rows']), int(cfg['columns'])
        desc = _lib.SxConfigDesc()
        desc.rows, desc.cols = self.rows, self.columns
        desc.max_turns, desc.usable_rows = int(cfg['max_turns']), int(cfg['initial_state_usable_rows'])
        amounts = piece_amounts_array(cfg['piece_amounts'])
        for i in range(13):
            desc.piece_amounts[i] = int(amounts[i])
        self._obst = np.ascontiguousarray(obstacle_map(cfg).reshape(-1), dtype=np.uint8)
        if normalize:
            self._cap_lut = np.ascontiguousarray((original_captured_lut if original else captured_lut)(cfg['piece_amounts']),
                                                 dtype=np.float32)
            self._recent_lut = np.ascontiguousarray(recent_moves_lut(), dtype=np.float32)
            self._unit_lut = np.ascontiguousarray(original_unit_lut() if original else unit_channel_lut(), dtype=np.float32)
            self._rank_lut = np.ascontiguousarray(original_rank_lut(), dtype=np.float32)
            self._po_rank_lut = np.ascontiguousarray(original_po_rank_lut(), dtype=np.float32)
        else:
            self._cap_lut = np.ascontiguousarray(np.tile(np.arange(9, dtype=np.float32), (12, 1)))
            self._recent_lut = np.arange(-3, 2, dtype=np.float32)
            self._unit_lut = np.asarray([0.0, 1.0], dtype=np.float32)
            self._rank_lut = np.arange(14, dtype=np.float32)
            self._po_rank_lut = np.arange(14, dtype=np.float32)
        desc.obs_channel_mode = _lib.SX_CHANNELS_ORIGINAL if original else _lib.SX_CHANNELS_EXTENDED
        desc.rank_lut = self._rank_lut.ctypes.data
        desc.po_rank_lut = self._po_rank_lut.ctypes.data
        desc.obstacles = self._obst.ctypes.data
        desc.captured_lut = self._cap_lut.ctypes.data
        desc.recent_lut = self._recent_lut.ctypes.data
        desc.unit_lut = self._unit_lut.ctypes.data
        desc.p2_rot180 = 1 if p2_rot180 else 0
        desc.capture_capacity = int(capture_capacity)
        desc.obs_dtype = desc_obs_dtype
        handle = C.c_void_p()
        _lib.check(self.lib.sx_config_create(C.byref(desc), C.byref(handle)), "sx_config_create")
        self._cfg = handle
        lay = _lib.SxLayout()
        _lib.check(self.lib.sx_config_layout(self._cfg, C.byref(lay)), "sx_config_layout")
        self.layout = lay
        self.cells = lay.cells
        self.spatial_channels = lay.spatial_channels
        self.po_channels, self.fo_channels = lay.po_channels, lay.fo_channels
        self.spatial_action_size = (self.rows, self.columns, lay.spatial_channels)
        self.action_size = lay.action_size

    def set_start_states(self, dense: Optional[torch.Tensor], num_envs: int = 0, env_base: int = 0):
        """Curriculum starts (curriculum_start_states_path, maenv:341-351 / 519-527, util:373-387): from now on ``reset`` and
        the auto-reset of ``step_all`` start every game from a uniformly drawn entry of ``dense`` (int64 [n, 34, R, C],
        the reference's state layout) with the turn counter at 0, this configuration's max_turns and a uniformly drawn
        player to move, instead of dealing setups.  ``None`` switches back.  Returns an int32 [num_envs] tensor that always
        holds the entry each env's current game came from (None when num_envs is 0)."""
        if dense is None:
            _lib.check(self.lib.sx_config_set_start_states(self._cfg, _lib.SxState(), 0, None, 0, 0), "sx_config_set_start_states")
            self._start_table = self._start_index = None
            return None
        dense = dense.to(self.device, dtype=torch.int64).clone()
        dense[:, 5, 0, 0] = 0                    # StateData.TURN_COUNT   (util:382)
        dense[:, 5, 1, 0] = int(self.game_version_config['max_turns'])  # StateData.MAX_TURNS (util:383)
        table = self.import_ref_state(dense)
        index = torch.zeros(num_envs, dtype=torch.int32, device=self.device) if num_envs else None
        _lib.check(self.lib.sx_config_set_start_states(self._cfg, table.as_struct(), table.num_envs,
                                                       index.data_ptr() if index is not None else None, int(env_base),
                                                       int(num_envs)),
                   "sx_config_set_start_states")
        self._start_table, self._start_index = table, index  # the library keeps raw pointers: keep the tensors alive
        return index

    def set_tuning(self, warps_per_block: int = -1, issue_point: int = -1, compact_movers: int = -1) -> None:
        """Result-preserving launch tuning of the warp-level kernel (sx_config_set_tuning; -1 keeps the built-in choice)."""
        _lib.check(self.lib.sx_config_set_tuning(self._cfg, int(warps_per_block), int(issue_point), int(compact_movers)),
                   "sx_config_set_tuning")

    def __del__(self):
        try:
            if getattr(self, "_cfg", None):
                self.lib.sx_config_destroy(self._cfg)
                self._cfg = None
        except Exception:  # noqa: BLE001
            pass

    # ---- buffers -------------------------------------------------------------------------------
    def alloc_state(self, num_envs: int) -> DeviceState:
        """the three state tensors are views of ONE allocation (one contiguous range to checkpoint or copy)"""
        d, lay = self.device, self.layout
        board_b, aux_b, cap_b = num_envs * lay.board_stride, num_envs * lay.aux_stride * 2, num_envs * lay.captured_stride * 2
        pad = lambda n: (n + 255) // 256 * 256  # noqa: E731
        buf = torch.zeros(pad(board_b) + pad(aux_b) + pad(cap_b), dtype=torch.uint8, device=d)
        board = buf[:board_b].view(num_envs, lay.board_stride)
        aux = buf[pad(board_b):pad(board_b) + aux_b].view(torch.int16).view(num_envs, lay.aux_stride)
        cap = buf[pad(board_b) + pad(aux_b):pad(board_b) + pad(aux_b) + cap_b].view(torch.int16).view(num_envs, lay.captured_stride)
        return DeviceState(board, aux, cap)

    def alloc_outputs(self, num_envs: int, partial=True, full=False, mask=True, sample=False, terminal=False) -> dict:
        """terminal=True adds the side buffers that receive BOTH players' observations of a game that ends during
        ``step_all`` (maenv:772-773): [B, 2, R, C, channels], index 0 = player +1's view; rows of games with done = 1"""
        d, R, Cc = self.device, self.rows, self.columns
        out = {
            "reward": torch.zeros(num_envs, dtype=torch.float32, device=d),
            "done": torch.zeros(num_envs, dtype=torch.uint8, device=d),
            "winner": torch.zeros(num_envs, dtype=torch.int8, device=d),
            "ending_invalid": torch.zeros(num_envs, dtype=torch.uint8, device=d),
            "illegal": torch.zeros(num_envs, dtype=torch.uint8, device=d),
            "player": torch.zeros(num_envs, dtype=torch.int8, device=d),
        }
        planes = []  # (name, shape, dtype, zero-filled)
        if partial:
            planes.append(("partial_obs", (num_envs, R, Cc, self.po_channels), self.obs_dtype, False))
        if full:
            planes.append(("full_obs", (num_envs, R, Cc, self.fo_channels), self.obs_dtype, False))
        if mask:
            planes.append(("valid_mask", (num_envs, R, Cc, self.spatial_channels), torch.uint8, False))
        if terminal and partial:
            planes.append(("terminal_partial_obs", (num_envs, 2, R, Cc, self.po_channels), self.obs_dtype, True))
        if terminal and full:
            planes.append(("terminal_full_obs", (num_envs, 2, R, Cc, self.fo_channels), self.obs_dtype, True))
        out.update(self._alloc_planes(planes))
        if sample:
            out["next_action"] = torch.zeros(num_envs, dtype=torch.int32, device=d)
        return out

    # Below one granule of compressible memory (2 MB on B200) compression rounds up more than it can save, and the
    # allocation and its synchronising free would dominate the small per-call buffers of the one-game API.
    _COMPRESSIBLE_MIN_BYTES = 2 << 20

    def _alloc_planes(self, planes) -> dict:
        """the observation / mask planes: torch tensors, or views of ONE library allocation (compressible where the
        device grants it) that the views keep alive"""
        size = lambda shape, dtype: int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()  # noqa: E731
        pad = lambda n: (n + 255) // 256 * 256  # noqa: E731
        total = sum(pad(size(shape, dtype)) for _, shape, dtype, _ in planes)
        if self.compressible_outputs is False or total < self._COMPRESSIBLE_MIN_BYTES:
            if planes:
                self.outputs_compressed = False
            return {name: (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=self.device)
                    for name, shape, dtype, zero in planes}
        alloc = DeviceAllocation(self.device, total, compressible=self._alloc_compressible)
        if self.compressible_outputs and not alloc.compressed:
            raise _lib.StrategoB200Error("compressible_outputs=True: device %s did not grant compressible memory"
                                         % self.device)
        self.outputs_compressed = alloc.compressed
        with torch.cuda.device(self.device):
            buf = torch.as_tensor(alloc, device=self.device)
        out, off = {}, 0
        for name, shape, dtype, zero in planes:
            n = size(shape, dtype)
            out[name] = buf[off:off + n].view(dtype).view(shape)
            if zero:
                out[name].zero_()
            off += pad(n)
        return out

    # False: the library's plain-memory path, the one a device without compression takes (the tests force it so)
    _alloc_compressible = True

    _OBS_OUTPUTS = ("partial_obs", "full_obs", "terminal_partial_obs", "terminal_full_obs")

    def _outputs_struct(self, out: dict) -> _lib.SxOutputs:
        s = _lib.SxOutputs()
        for name, _ in _lib.SxOutputs._fields_:
            t = out.get(name)
            if t is not None:
                assert t.is_cuda and t.is_contiguous(), name
                if name in self._OBS_OUTPUTS and t.dtype != self.obs_dtype:
                    raise ValueError("%s is %s; this engine writes %s observations" % (name, t.dtype, self.obs_dtype))
                setattr(s, name, t.data_ptr())
        return s

    def upload_setups(self, table: np.ndarray) -> torch.Tensor:
        table = np.ascontiguousarray(table, dtype=np.uint8)
        assert table.ndim == 2 and table.shape[1] == self.layout.setup_len, (table.shape, self.layout.setup_len)
        return torch.from_numpy(table).to(self.device)

    # ---- operations ----------------------------------------------------------------------------
    def reset(self, state: DeviceState, seed: int = 0, env_base: int = 0, reset_mask: Optional[torch.Tensor] = None,
              setups: Optional[torch.Tensor] = None, setup_idx: Optional[torch.Tensor] = None, shuffle: bool = False,
              same_setup: bool = False, repeat_other_side: bool = False):
        """same_setup: every game of an env starts from its first draw (maenv:352-354); repeat_other_side: every second
        game of an env repeats the previous initial position from the other side (maenv:530-534)"""
        flags = ((_lib.SX_RESET_RANDOM_SHUFFLE if shuffle else 0) | (_lib.SX_SAME_SETUP if same_setup else 0) |
                 (_lib.SX_REPEAT_OTHER_SIDE if repeat_other_side else 0))
        if setup_idx is not None:
            assert setup_idx.dtype == torch.int32 and setup_idx.shape == (state.num_envs, 2) and setup_idx.is_contiguous()
        if reset_mask is not None:
            assert reset_mask.dtype == torch.uint8 and reset_mask.is_contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_reset(self._cfg, state.as_struct(), state.num_envs, env_base, _ptr(reset_mask),
                                         _ptr(setups), 0 if setups is None else setups.shape[0], _ptr(setup_idx),
                                         seed & (2 ** 64 - 1), flags, _stream()), "sx_reset")

    def import_ref_state(self, dense: torch.Tensor, player: Optional[torch.Tensor] = None,
                         state: Optional[DeviceState] = None, check: bool = True) -> DeviceState:
        """dense: int64 [B, 34, R, C] in the reference's layout (impl:16-60); player: int8 [B] (+1/-1)."""
        dense = dense.to(self.device, dtype=torch.int64).contiguous()
        B = dense.shape[0]
        assert dense.shape == (B, NUM_STATE_LAYERS, self.rows, self.columns), dense.shape
        if player is not None:
            player = player.to(self.device, dtype=torch.int8).contiguous()
        if state is None:
            state = self.alloc_state(B)
        status = torch.zeros(B, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_import_ref_state(self._cfg, state.as_struct(), B, dense.data_ptr(), _ptr(player),
                                                    status.data_ptr(), _stream()), "sx_import_ref_state")
        if check and bool(status.any().item()):
            bad = torch.nonzero(status).flatten().tolist()[:8]
            raise ValueError("state(s) %s cannot be represented by the compact device layout (not reachable by play)"
                             % bad)
        return state

    # torch integer dtypes a viewer tensor may have (bool is not one)
    _VIEWER_DTYPES = (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8)

    def sample_hidden_states(self, state: DeviceState, n_samples: int = 1, viewer: Optional[torch.Tensor] = None,
                             seed: int = 0, draw: int = 0, env_base: int = 0, check: bool = True) -> DeviceState:
        """Determinization (sx_sample_hidden_states): ``n_samples`` complete game states per game that agree with what
        the viewer knows.  The opponent's unrevealed pieces are re-placed uniformly at random among the placements that
        keep the multiset of their codes and put no flag or bomb on a piece that has moved; everything else is copied.
        viewer: None (the player to move) or an integer tensor [B], 1 = player +1, anything else = player -1.
        Returns a new DeviceState of B * n_samples rows in this engine's strides, row b * n_samples + k = sample k of
        game b, ready for observe / step / step_all / export_ref_state.  Sample k of a game depends only on (seed, draw,
        env_base + b, k).  check=True: a game in which more flags and bombs are hidden than unmoved hidden pieces exist
        (no placement; only an imported state can be so) raises ValueError naming the games; with check=False its rows
        are plain copies."""
        if isinstance(n_samples, bool) or not isinstance(n_samples, (int, np.integer)) or not 1 <= n_samples < 1 << 24:
            raise ValueError("n_samples must be an integer in [1, 2^24), not %r" % (n_samples,))
        B = state.num_envs
        if viewer is not None:
            self._check_viewer(viewer, B)
            viewer = viewer.to(self.device, dtype=torch.int8).contiguous()
        n_samples = int(n_samples)
        out = self.alloc_state(B * n_samples)
        status = torch.zeros(B, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_sample_hidden_states(self._cfg, state.as_struct(), B, int(env_base), _ptr(viewer),
                                                        n_samples, seed & (2 ** 64 - 1), int(draw) & 0xffffffff,
                                                        out.as_struct(), status.data_ptr(), _stream()),
                       "sx_sample_hidden_states")
        if check and bool(status.any().item()):
            bad = torch.nonzero(status).flatten().tolist()[:8]
            raise ValueError("game(s) %s hide more flags and bombs than unmoved pieces: no consistent placement exists "
                             "(not reachable by play)" % bad)
        return out

    def _check_viewer(self, viewer, B: int) -> None:
        """ValueError unless ``viewer`` is an integer tensor of shape (B,) (checked on the host)"""
        if not isinstance(viewer, torch.Tensor) or viewer.dtype not in self._VIEWER_DTYPES or tuple(viewer.shape) != (B,):
            raise ValueError("viewer must be None or an integer tensor of shape (%d,), not %s" % (
                B, "%s %s" % (viewer.dtype, tuple(viewer.shape)) if isinstance(viewer, torch.Tensor) else type(viewer).__name__))

    def _check_tensor(self, name, t, dtypes, shapes) -> None:
        """ValueError unless ``t`` is a contiguous tensor of one of ``dtypes`` and one of ``shapes`` on this engine's
        device (checked on the host, before any device is touched)"""
        if (not isinstance(t, torch.Tensor) or t.dtype not in dtypes or t.shape not in shapes or not t.is_contiguous()
                or t.device != self.device):
            raise ValueError("%s must be a contiguous %s tensor of shape %s on %s, not %s" % (
                name, " / ".join(map(str, dtypes)), " or ".join(map(str, shapes)), self.device,
                "%s %s on %s" % (t.dtype, tuple(t.shape), t.device) if isinstance(t, torch.Tensor) else type(t).__name__))

    def _check_state(self, state) -> None:
        """ValueError unless ``state`` is a DeviceState of contiguous tensors in this engine's dtypes, strides and
        device"""
        lay = self.layout
        if not isinstance(state, DeviceState):
            raise ValueError("state must be a DeviceState, not %s" % type(state).__name__)
        B = state.num_envs
        for name, t, dtype, width in (("state.board", state.board, torch.uint8, lay.board_stride),
                                      ("state.aux", state.aux, torch.int16, lay.aux_stride),
                                      ("state.captured", state.captured, torch.int16, lay.captured_stride)):
            self._check_tensor(name, t, (dtype,), ((B, width),))

    @staticmethod
    def _root_player(state: DeviceState) -> torch.Tensor:
        """int8 [B]: the player to move in each game (+1 / -1), from aux_pack's to_move bit"""
        return torch.where(((state.aux[:, 2] >> 4) & 1) == 0, 1, -1).to(torch.int8)

    def expand_moves(self, state: DeviceState) -> "Expansion":
        """The children of every game (sx_count_moves + sx_expand_moves): one per legal move of the player to move, in
        ascending flat spatial index (that player's frame, the index step / step_all / sample_policy take).  Child j of
        game b is row offsets[b] + j of every field and equals, byte for byte, what ``step`` (spatial actions, no flags)
        makes of a copy of game b with action actions[row]: state rows and the reward, done, winner, ending_invalid,
        illegal and player it returns.  A finished game or a stuck player has no children.  ``state`` is not written.
        Reading the number of children back to size the outputs is ONE host synchronisation per call."""
        self._check_state(state)
        B = state.num_envs
        d = self.device
        counts = torch.empty(B, dtype=torch.int32, device=d)
        offsets = torch.zeros(B + 1, dtype=torch.int64, device=d)
        with torch.cuda.device(d):
            _lib.check(self.lib.sx_count_moves(self._cfg, state.as_struct(), B, counts.data_ptr(), _stream()),
                       "sx_count_moves")
            torch.cumsum(counts, 0, dtype=torch.int64, out=offsets[1:])
            T = int(offsets[-1].item())  # the host synchronisation
            out = self.alloc_state(T)
            scalars = self.alloc_outputs(T, partial=False, full=False, mask=False)
            actions = torch.empty(T, dtype=torch.int32, device=d)
            _lib.check(self.lib.sx_expand_moves(self._cfg, state.as_struct(), B, offsets.data_ptr(), T, out.as_struct(),
                                                actions.data_ptr(), self._outputs_struct(scalars), _stream()),
                       "sx_expand_moves")
            parent = torch.repeat_interleave(torch.arange(B, device=d), counts, output_size=T)
        return Expansion(states=out, actions=actions, parent=parent, offsets=offsets, **scalars)

    def playout(self, state: DeviceState, max_plies: Optional[int] = None, seed: int = 0, env_base: int = 0) -> "Playout":
        """Random playouts (sx_playout): every game of ``state`` is played on, in place, with uniformly random legal
        moves until it ends or ``max_plies`` plies have been played (None: to the end).  The move of each ply is the
        draw ``step_all(..., sample_next=True, seed=seed, env_base=env_base)`` makes for the state before that ply, so a
        playout of n plies equals, byte for byte, n such chained steps (without auto-reset) stopped at the first that
        reports done, and continues the chain of a caller's last ``step_all`` with that seed.  A game over at entry plays
        0 plies and is not written; a player to move without a legal move (only an imported state can be so) loses, as
        with the noop action.  Returns the plies played and, per game, the reward, done, winner, ending_invalid, illegal
        and player as the step that ended the game reported them.  No host synchronisation."""
        if max_plies is not None and (isinstance(max_plies, bool) or not isinstance(max_plies, (int, np.integer))
                                      or not 0 <= max_plies < 1 << 31):
            raise ValueError("max_plies must be None or an integer in [0, 2^31), not %r" % (max_plies,))
        self._check_state(state)
        B = state.num_envs
        d = self.device
        plies = torch.empty(B, dtype=torch.int32, device=d)
        scalars = self.alloc_outputs(B, partial=False, full=False, mask=False)
        with torch.cuda.device(d):
            _lib.check(self.lib.sx_playout(self._cfg, state.as_struct(), B, int(env_base),
                                           (1 << 31) - 1 if max_plies is None else int(max_plies), seed & (2 ** 64 - 1),
                                           plies.data_ptr(), self._outputs_struct(scalars), _stream()), "sx_playout")
        return Playout(plies=plies, **scalars)

    @staticmethod
    def _check_int(name, value, lo, hi, allow_none=False):
        """ValueError unless ``value`` is an integer (not a bool) in [lo, hi] (or None where allowed)"""
        if value is None and allow_none:
            return
        if isinstance(value, bool) or not isinstance(value, (int, np.integer)) or not lo <= value <= hi:
            raise ValueError("%s must be %san integer in [%d, %d], not %r" % (
                name, "None or " if allow_none else "", lo, hi, value))

    @staticmethod
    def _check_float(name, value, lo=None, hi=None):
        """ValueError unless ``value`` is a real number (not a bool) that is finite in float32 (and >= lo, <= hi)"""
        if type(value) is float:  # the common case, without numpy's error-state context (a few us per call)
            # 2^128 - 2^103, half an ulp above FLT_MAX: the least magnitude float32 rounding sends to infinity
            bad = (not abs(value) < 3.4028235677973366e38 or (lo is not None and not value >= lo)
                   or (hi is not None and not value <= hi))
        else:
            with np.errstate(over="ignore"):
                bad = (isinstance(value, bool) or not isinstance(value, (int, float, np.integer, np.floating))
                       or not np.isfinite(np.float32(value)) or (lo is not None and not value >= lo)
                       or (hi is not None and not value <= hi))
        if bad:
            raise ValueError("%s must be a finite number%s%s (in float32), not %r" % (
                name, "" if lo is None else " >= %g" % lo, "" if hi is None else " <= %g" % hi, value))

    def search(self, state: DeviceState, iterations: int, max_nodes: Optional[int] = None,
               max_plies: Optional[int] = None, c_explore: float = 1.0, seed: int = 0, env_base: int = 0) -> "SearchTree":
        """Monte Carlo tree search (sx_search), one tree per game of ``state`` with that game as its root, all in one
        launch.  Each of the ``iterations`` iterations descends from the root (the first unvisited child, else the child
        of best PUCT score with a uniform prior, q + c_explore * sqrt(N_parent) / (1 + N_child), q seen from the
        player to move), expands a leaf into all its legal moves (ascending flat spatial index, the ``expand_moves``
        action list) while the pool of ``max_nodes`` nodes has room, scores the state reached by its outcome or a random
        playout of at most ``max_plies`` plies (None: to the end), and adds the score to N and W along the path.
        max_nodes=None: 1 + 32 * iterations.  The tree depends only on (seed, env_base + b, the root, iterations,
        max_nodes, max_plies, c_explore); ``state`` is not written.  Returns a SearchTree; ``root_stats()`` gives the
        root children's visits and values in the valid-mask shape.  No host synchronisation."""
        self._check_int("iterations", iterations, 0, 1 << 24)
        if max_nodes is None and not isinstance(iterations, bool) and isinstance(iterations, (int, np.integer)):
            max_nodes = 1 + 32 * int(iterations)
        self._check_int("max_nodes", max_nodes, 1, (1 << 31) - 1)
        self._check_int("max_plies", max_plies, 0, (1 << 31) - 1, allow_none=True)
        self._check_float("c_explore", c_explore, lo=0)
        self._check_state(state)
        B, M = state.num_envs, int(max_nodes)
        d = self.device
        f = [torch.empty((B, M), dtype=torch.int32, device=d) for _ in range(6)]
        used = torch.empty(B, dtype=torch.int32, device=d)
        tree = _lib.SxTree(*(t.data_ptr() for t in f), used.data_ptr())
        with torch.cuda.device(d):
            _lib.check(self.lib.sx_search(self._cfg, state.as_struct(), B, int(env_base), int(iterations), M,
                                          (1 << 31) - 1 if max_plies is None else int(max_plies), float(c_explore),
                                          seed & (2 ** 64 - 1), tree, _stream()), "sx_search")
            root_player = self._root_player(state)
        return SearchTree(*f, used=used, root_player=root_player,
                          mask_shape=(self.rows, self.columns, self.spatial_channels))

    # ---- guided search: PUCT select and backup on the device, leaves evaluated by the caller -------------------------
    def guided_tree(self, roots: DeviceState, max_nodes: int) -> "SearchTree":
        """An empty guided tree per game of ``roots`` (sx_guided_select / sx_guided_backup): the root alone, used = 1,
        N = 0, W = 0, parent = first_child = -1, n_children = 0, action = -1, P = 1; ``value`` and ``prior`` are float32
        [B, max_nodes], the other node fields int32.  Written with torch fills, no host synchronisation."""
        self._check_int("max_nodes", max_nodes, 1, (1 << 31) - 1)
        self._check_state(roots)
        B, M, d = roots.num_envs, int(max_nodes), self.device
        visits, parent, first_child, n_children, action = (torch.empty((B, M), dtype=torch.int32, device=d)
                                                           for _ in range(5))
        value, prior = (torch.empty((B, M), dtype=torch.float32, device=d) for _ in range(2))
        for t, x in ((visits, 0), (value, 0.0), (parent, -1), (first_child, -1), (n_children, 0), (action, -1),
                     (prior, 1.0)):
            t[:, 0].fill_(x)
        used = torch.ones(B, dtype=torch.int32, device=d)
        return SearchTree(visits, value, parent, first_child, n_children, action, used=used,
                          root_player=self._root_player(roots),
                          mask_shape=(self.rows, self.columns, self.spatial_channels), prior=prior)

    def _check_guided_tree(self, tree, B: int) -> int:
        """max_nodes of ``tree``; ValueError unless it is a guided SearchTree of B trees on this engine's device"""
        if not isinstance(tree, SearchTree) or not isinstance(tree.prior, torch.Tensor):
            raise ValueError("tree must be a SearchTree made by guided_tree, not %s" % type(tree).__name__)
        M = tree.visits.shape[1] if isinstance(tree.visits, torch.Tensor) and tree.visits.dim() == 2 else -1
        i32, f32, nodes = (torch.int32,), (torch.float32,), ((B, M),)
        for name, t, dtypes, shapes in (("tree.visits", tree.visits, i32, nodes), ("tree.value", tree.value, f32, nodes),
                                        ("tree.parent", tree.parent, i32, nodes),
                                        ("tree.first_child", tree.first_child, i32, nodes),
                                        ("tree.n_children", tree.n_children, i32, nodes),
                                        ("tree.action", tree.action, i32, nodes), ("tree.prior", tree.prior, f32, nodes),
                                        ("tree.used", tree.used, i32, ((B,),))):
            self._check_tensor(name, t, dtypes, shapes)
        if M < 1:
            raise ValueError("tree must have max_nodes >= 1, not %d" % M)
        return M

    def _guided_struct(self, tree) -> "_lib.SxGuidedTree":
        return _lib.SxGuidedTree(*(getattr(tree, n).data_ptr() for n, _ in _lib.SxGuidedTree._fields_))

    def guided_select(self, roots: DeviceState, tree: "SearchTree", c_puct: float = 1.25, fpu: float = 0.0,
                      leaves_per_tree: int = 1, virtual_loss: float = 1.0) -> "Leaves":
        """``leaves_per_tree`` = L leaves per tree (sx_guided_select_many): descend from the root of ``tree`` (the game of
        ``roots``) by the PUCT score q + c_puct * P * sqrt(N_parent) / (1 + N), q = the mean value from the mover's side
        or ``fpu`` for an unvisited child, ties to the lowest index, to the first node without children or whose state
        is over.  Leaves j = 0 .. L-1 of a tree are chosen in order, each from the root: the paths of leaves 0 .. j-1
        count as pending visits V (N + V in place of N, and each pending visit takes ``virtual_loss`` from the mover's
        value, q = (sigma * W - virtual_loss * V) / (N + V)).  L = 1 is the one-leaf select exactly.  Returns the
        leaves' states (ready for ``observe``, ``valid_mask``, ``export_ref_state``), node indices and kinds (LEAF_EVAL,
        LEAF_OVER, LEAF_STUCK), B * L rows, leaf j of tree b at row b * L + j.  Neither ``roots`` nor the tree's node
        fields are written, so two selects without a backup between them return the same leaves.  L in [1, 1024];
        virtual_loss finite in [0, 2^24].  The first call with L > 1 on a tree gives it ``tree.inflight`` (int32
        [B, max_nodes] zeros, all zero again after every select), so capture a CUDA graph of L > 1 rounds after one
        warm-up round.  No host synchronisation."""
        self._check_state(roots)
        B = roots.num_envs
        M = self._check_guided_tree(tree, B)
        self._check_float("c_puct", c_puct, lo=0)
        self._check_float("fpu", fpu)
        self._check_int("leaves_per_tree", leaves_per_tree, 1, _lib.SX_GUIDED_MAX_LEAVES)
        self._check_float("virtual_loss", virtual_loss, lo=0, hi=2 ** 24)
        if tree.inflight is not None:
            self._check_tensor("tree.inflight", tree.inflight, (torch.int32,), ((B, M),))
        L = int(leaves_per_tree)
        if L > 1 and tree.inflight is None:
            tree.inflight = torch.zeros((B, M), dtype=torch.int32, device=self.device)
        leaves = Leaves(self.alloc_state(B * L), torch.empty(B * L, dtype=torch.int32, device=self.device),
                        torch.empty(B * L, dtype=torch.int8, device=self.device), per_tree=L)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_guided_select_many(self._cfg, roots.as_struct(), B, self._guided_struct(tree), M,
                                                      float(c_puct), float(fpu), L, float(virtual_loss),
                                                      _ptr(tree.inflight), leaves.states.as_struct(),
                                                      leaves.node.data_ptr(), leaves.kind.data_ptr(), _stream()),
                       "sx_guided_select_many")
        return leaves

    def guided_backup(self, tree: "SearchTree", leaves: "Leaves", logits: torch.Tensor, values: torch.Tensor) -> None:
        """Expand and back up the leaves of the last ``guided_select`` (sx_guided_backup_many), L = leaves.per_tree
        per tree.  logits: float32, bfloat16 or float16 [B * L, R, C, A] (or [B * L, R * C * A]) in the layout of
        ``sample_policy`` (the leaf's player-to-move frame); values: float32 [B * L], the leaf's value from the side of
        its player to move.  The leaves of a tree are taken in order: an evaluable leaf whose node has no children yet
        gets its legal moves as children (the ``expand_moves`` order) with the softmax of its logits over them as
        priors, if the pool has room; then the leaf and its ancestors get N += 1 and W += the value in absolute terms
        (a finished leaf's outcome, or a loss for a stuck player to move).  A node several leaves reached is expanded
        once, by the first of them, and each of them backs up its own value.  No host synchronisation."""
        if not isinstance(leaves, Leaves):
            raise ValueError("leaves must be the Leaves guided_select returned, not %s" % type(leaves).__name__)
        self._check_int("leaves.per_tree", leaves.per_tree, 1, _lib.SX_GUIDED_MAX_LEAVES)
        self._check_state(leaves.states)
        L = int(leaves.per_tree)
        rows = leaves.states.num_envs
        if rows % L:
            raise ValueError("leaves must have a multiple of leaves.per_tree = %d rows, not %d" % (L, rows))
        B = rows // L
        M = self._check_guided_tree(tree, B)
        self._check_tensor("leaves.node", leaves.node, (torch.int32,), ((rows,),))
        self._check_tensor("leaves.kind", leaves.kind, (torch.int8,), ((rows,),))
        self._check_tensor("logits", logits, tuple(OBS_DTYPES),
                           ((rows,) + tuple(self.spatial_action_size), (rows, self.layout.spatial_actions)))
        self._check_tensor("values", values, (torch.float32,), ((rows,),))
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_guided_backup_many(self._cfg, leaves.states.as_struct(), B, self._guided_struct(tree),
                                                      M, L, leaves.node.data_ptr(), leaves.kind.data_ptr(),
                                                      logits.data_ptr(), OBS_DTYPES[logits.dtype], values.data_ptr(),
                                                      _stream()),
                       "sx_guided_backup_many")

    def state_keys(self, state: DeviceState, info_set: bool = False, viewer: Optional[torch.Tensor] = None) -> torch.Tensor:
        """64-bit keys that identify positions (sx_state_keys), int64 [B]: the uint64 key bits viewed as int64, so that
        ``torch.unique`` and ``torch.isin`` take them directly.
        info_set=False: the key of each game as ``export_ref_state`` exports it (dense state and player to move).  Equal
        exports give equal keys; the episode counter, board padding and the order of the capture list do not count.
        Different exports collide with probability about 2^-64 per pair (n states: about n^2 / 2^65).
        info_set=True: the key of what ``viewer`` knows: the same, but the opponent's unrevealed pieces count as UNKNOWN
        whatever their true rank, and the viewer is part of the key.  viewer: None (the player to move) or an integer
        tensor [B], 1 = player +1, anything else = player -1, as for ``sample_hidden_states``; every state that call
        draws for a viewer has its source's information-set key for that viewer.
        Keys depend on the position alone (no seed, no env_base), so tables can outlive a call and a process.  No host
        synchronisation."""
        self._check_state(state)
        if not isinstance(info_set, bool):
            raise ValueError("info_set must be True or False, not %r" % (info_set,))
        B = state.num_envs
        if viewer is not None:
            if not info_set:
                raise ValueError("viewer is only taken with info_set=True")
            self._check_viewer(viewer, B)
            viewer = viewer.to(self.device, dtype=torch.int8).contiguous()
        keys = torch.empty(B, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_state_keys(self._cfg, state.as_struct(), B, _ptr(viewer),
                                              _lib.SX_KEY_INFOSET if info_set else _lib.SX_KEY_STATE, keys.data_ptr(),
                                              _stream()), "sx_state_keys")
        return keys

    def export_ref_state(self, state: DeviceState):
        B = state.num_envs
        dense = torch.empty((B, NUM_STATE_LAYERS, self.rows, self.columns), dtype=torch.int64, device=self.device)
        player = torch.empty(B, dtype=torch.int8, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_export_ref_state(self._cfg, state.as_struct(), B, dense.data_ptr(),
                                                    player.data_ptr(), _stream()), "sx_export_ref_state")
        return dense, player

    def export_perspective_state(self, state: DeviceState, viewer: Optional[torch.Tensor] = None) -> torch.Tensor:
        """int64 [B, 34, R, C]: each game as `viewer[b]` (+1/-1; default: absolute frame) sees it (impl:646-675)."""
        B = state.num_envs
        dense = torch.empty((B, NUM_STATE_LAYERS, self.rows, self.columns), dtype=torch.int64, device=self.device)
        if viewer is not None:
            viewer = viewer.to(self.device, dtype=torch.int8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_export_perspective_state(self._cfg, state.as_struct(), B, _ptr(viewer),
                                                            dense.data_ptr(), _stream()), "sx_export_perspective_state")
        return dense

    def valid_mask(self, state: DeviceState, player: Optional[torch.Tensor] = None, one_d: bool = False) -> torch.Tensor:
        B = state.num_envs
        if one_d:
            mask = torch.empty((B, self.action_size), dtype=torch.uint8, device=self.device)
        else:
            mask = torch.empty((B,) + self.spatial_action_size, dtype=torch.uint8, device=self.device)
        if player is not None:
            player = player.to(self.device, dtype=torch.int8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_valid_mask(self._cfg, state.as_struct(), B, _ptr(player),
                                              _lib.SX_ACTION_1D if one_d else _lib.SX_ACTION_SPATIAL, mask.data_ptr(),
                                              _stream()), "sx_valid_mask")
        return mask

    def observe(self, state: DeviceState, player: Optional[torch.Tensor] = None, out: Optional[dict] = None,
                partial=True, full=True, mask=True) -> dict:
        if out is None:
            out = self.alloc_outputs(state.num_envs, partial=partial, full=full, mask=mask)
        if player is not None:
            player = player.to(self.device, dtype=torch.int8).contiguous()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_observe(self._cfg, state.as_struct(), state.num_envs, _ptr(player),
                                           self._outputs_struct(out), _stream()), "sx_observe")
        return out

    def step(self, state: DeviceState, actions: torch.Tensor, one_d: bool = False, allow_piece_oscillation=False,
             out: Optional[dict] = None) -> dict:
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.shape == (state.num_envs,)
        if out is None:
            out = self.alloc_outputs(state.num_envs, partial=False, full=False, mask=False)
        flags = _lib.SX_ALLOW_OSCILLATION if allow_piece_oscillation else 0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_step(self._cfg, state.as_struct(), state.num_envs, actions.data_ptr(),
                                        _lib.SX_ACTION_1D if one_d else _lib.SX_ACTION_SPATIAL, flags,
                                        self._outputs_struct(out), _stream()), "sx_step")
        return out

    def step_all(self, state: DeviceState, actions: torch.Tensor, out: dict, one_d: bool = False, env_base: int = 0,
                 auto_reset: bool = False, sample_next: bool = False, allow_piece_oscillation: bool = False,
                 setups: Optional[torch.Tensor] = None, shuffle: bool = False, seed: int = 0,
                 stats: Optional[torch.Tensor] = None, baseline_kernel: bool = False, same_setup: bool = False,
                 repeat_other_side: bool = False) -> dict:
        """baseline_kernel=True runs the general warp-per-game kernel even where a specialised kernel is eligible
        (identical results; the cross-kernel parity tests use it)."""
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.shape == (state.num_envs,)
        flags = ((_lib.SX_AUTO_RESET if auto_reset else 0) | (_lib.SX_SAMPLE_NEXT if sample_next else 0) |
                 (_lib.SX_ALLOW_OSCILLATION if allow_piece_oscillation else 0) |
                 (_lib.SX_RESET_RANDOM_SHUFFLE if shuffle else 0) | (_lib.SX_KERNEL_BASELINE if baseline_kernel else 0) |
                 (_lib.SX_SAME_SETUP if same_setup else 0) | (_lib.SX_REPEAT_OTHER_SIDE if repeat_other_side else 0))
        if stats is not None:
            assert stats.dtype == torch.int64 and stats.numel() >= 8
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_step_all(self._cfg, state.as_struct(), state.num_envs, env_base, actions.data_ptr(),
                                            _lib.SX_ACTION_1D if one_d else _lib.SX_ACTION_SPATIAL, flags,
                                            _ptr(setups), 0 if setups is None else setups.shape[0],
                                            seed & (2 ** 64 - 1), self._outputs_struct(out), _ptr(stats), _stream()),
                       "sx_step_all")
        return out

    def sample_valid(self, mask: torch.Tensor, seed: int = 0, step: int = 0, env_base: int = 0) -> torch.Tensor:
        B = mask.shape[0]
        flat = mask.reshape(B, -1)
        assert flat.dtype == torch.uint8 and flat.is_contiguous()
        actions = torch.empty(B, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_sample_valid(flat.data_ptr(), B, flat.shape[1], env_base, seed & (2 ** 64 - 1),
                                                step & 0xffffffff, actions.data_ptr(), _stream()), "sx_sample_valid")
        return actions

    def sample_logits(self, logits: torch.Tensor, mask: torch.Tensor, seed: int = 0, step: int = 0, env_base: int = 0,
                      temperature: float = 1.0, return_logprob: bool = False):
        """Masked categorical sampling: actions[b] ~ softmax(logits[b] / temperature) over mask[b] != 0
        (replaces the CPU chooser of examples/basic_game_loop.py:6-32).  logits: float32 / bfloat16 / float16
        [B, n_actions] (any trailing shape that flattens to it); mask: uint8, same number of entries."""
        B = mask.shape[0]
        flat_mask = mask.reshape(B, -1)
        flat_logits = logits.reshape(B, -1)
        assert flat_mask.dtype == torch.uint8 and flat_mask.is_contiguous() and flat_logits.is_contiguous()
        assert flat_logits.shape == flat_mask.shape, (flat_logits.shape, flat_mask.shape)
        dtype = OBS_DTYPES[flat_logits.dtype]
        actions = torch.empty(B, dtype=torch.int32, device=self.device)
        logprob = torch.empty(B, dtype=torch.float32, device=self.device) if return_logprob else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_sample_logits(flat_logits.data_ptr(), dtype, flat_mask.data_ptr(), B,
                                                 flat_mask.shape[1], env_base, seed & (2 ** 64 - 1), step & 0xffffffff,
                                                 float(temperature), actions.data_ptr(), _ptr(logprob), _stream()),
                       "sx_sample_logits")
        return (actions, logprob) if return_logprob else actions

    def sample_policy(self, state: DeviceState, logits: torch.Tensor, seed: int = 0, step: int = 0, env_base: int = 0,
                      temperature: float = 1.0, return_logprob: bool = False):
        """The draw of ``sample_logits`` taken from the game state instead of a mask (sx_sample_policy): the valid
        entries of the player to move are regenerated from the ~0.3 KB compact state, so the 3.7 KB mask row is never
        re-read.  Same Philox key => same action as ``sample_logits`` on that state's mask."""
        B = state.num_envs
        flat_logits = logits.reshape(B, -1)
        assert flat_logits.is_contiguous() and flat_logits.shape[1] == self.layout.spatial_actions, flat_logits.shape
        dtype = OBS_DTYPES[flat_logits.dtype]
        actions = torch.empty(B, dtype=torch.int32, device=self.device)
        logprob = torch.empty(B, dtype=torch.float32, device=self.device) if return_logprob else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_sample_policy(self._cfg, state.as_struct(), B, env_base, flat_logits.data_ptr(), dtype,
                                                 seed & (2 ** 64 - 1), step & 0xffffffff, float(temperature),
                                                 actions.data_ptr(), _ptr(logprob), _stream()), "sx_sample_policy")
        return (actions, logprob) if return_logprob else actions

    def heuristic_rewards(self, state: DeviceState, actions: torch.Tensor, reward_matrix: torch.Tensor,
                          one_d: bool = False) -> torch.Tensor:
        """impl:854-891 batched: reward_matrix[mover's rank at start, opponent's rank at end] of the action each game
        is about to play (call before the step).  reward_matrix: float32 [13, 13]."""
        assert actions.dtype == torch.int32 and actions.is_contiguous() and actions.shape == (state.num_envs,)
        matrix = reward_matrix.to(self.device, dtype=torch.float32).contiguous()
        assert matrix.shape == (13, 13), matrix.shape
        rewards = torch.empty(state.num_envs, dtype=torch.float32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_heuristic_rewards(self._cfg, state.as_struct(), state.num_envs, actions.data_ptr(),
                                                     _lib.SX_ACTION_1D if one_d else _lib.SX_ACTION_SPATIAL,
                                                     matrix.data_ptr(), rewards.data_ptr(), _stream()),
                       "sx_heuristic_rewards")
        return rewards

    def launch_info(self, partial=True, full=False, mask=True) -> dict:
        """launch shape of sx_step_all for these outputs, in compressible memory when the last ``alloc_outputs`` got it"""
        info = _lib.SxLaunchInfo()
        obs = (1 if partial else 0) | (2 if full else 0) | (4 if mask else 0) | (8 if self.outputs_compressed else 0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.sx_step_all_launch_info(self._cfg, obs, C.byref(info)), "sx_step_all_launch_info")
        return {n: getattr(info, n) for n, _ in _lib.SxLaunchInfo._fields_}
