// sx_keys.cu -- 64-bit keys that identify positions, for transposition tables and information-set search.
//
// Only the engine knows which bytes of the compact state are part of the game: the aux episode counter is an RNG stream
// number, board padding is not a cell, the capture list is kept in capture order, and which rank nibbles a player
// cannot see is the determinization rule of sx_hidden.cu.  So the key is defined on what sx_export_ref_state exports,
// the dense int64 [34, R, C] state plus the player to move.  Contract (include/stratego_b200.h, DESIGN.md §3.3):
//
//   state key = XOR of zobrist(c, l, x) over every non-zero dense entry x at (layer l, cell c), layers 0-1 and 3-33
//   (layer 2, the obstacles, is fixed by the configuration), and zobrist(0, KEY_LAYER_PLAYER, player to move +1 / -1);
//   information-set key for viewer v: the same after replacing, on every hidden cell (as sx_sample_hidden_states
//   defines it), the opponent's true rank in layer opp with its PO-layer entry 3 + opp (UNKNOWN, 13), plus
//   zobrist(0, KEY_LAYER_VIEWER, v);
//   zobrist(c, l, x) = words 0 | 1 << 32 of Philox4x32-10, key (KEY_PHILOX_LO, KEY_PHILOX_HI), counter (c, l, uint32(x),
//   RNG_KEYS).
//
// One warp per game on every board.  The dense features are derived from the compact state in registers: a ballot pass
// lists the occupied cells (cell | byte << 8) in the warp's shared slice, then feature slot f of the game goes to lane
// f mod 32: slots [0, n) the true-rank layer of occupied cell f, [n, 2n) its PO layer, [2n, 3n) its still layer,
// then the data layer (5 entries), the recent moves (4), the player, the viewer and one slot per capture entry.  A slot
// whose entry is zero computes its Philox block and drops it, so all lanes stay converged; the lanes' words are folded
// with __reduce_xor_sync.  Philox blocks per lane and game, ceil(slots / 32): 2.0 on de-phased Barrage, 7.9 on Standard.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int KEYS_WARPS = 8;  // warps per block
constexpr uint32_t KEY_PHILOX_LO = 0x53545241u, KEY_PHILOX_HI = 0x5445474fu;  // "STRA", "TEGO"
constexpr uint32_t KEY_LAYER_PLAYER = SX_NUM_STATE_LAYERS, KEY_LAYER_VIEWER = SX_NUM_STATE_LAYERS + 1;
constexpr int KEY_EXTRA_SLOTS = 11;  // data layer 5, recent moves 4, player 1, viewer 1

__device__ __forceinline__ uint64_t zobrist(uint32_t cell, uint32_t layer, uint32_t value)
{
    const uint4 r = philox4x32_10(make_uint4(cell, layer, value, RNG_KEYS), make_uint2(KEY_PHILOX_LO, KEY_PHILOX_HI));
    return uint64_t(r.x) | (uint64_t(r.y) << 32);
}

__global__ void __launch_bounds__(KEYS_WARPS * 32) sx_state_keys_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
    long long num_envs, const int8_t *viewer, int infoset, uint64_t *keys)
{
    __shared__ uint16_t occ_all[KEYS_WARPS][256];  // occupied cells of the warp's game: cell | cell byte << 8
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint16_t *occ = occ_all[warp];
    const uint32_t lt = (1u << lane) - 1u;

    for (long long b = (long long)blockIdx.x * KEYS_WARPS + warp; b < num_envs; b += (long long)gridDim.x * KEYS_WARPS) {
        Aux a;
        unpack(*reinterpret_cast<const uint4 *>(aux + b * 8), a);
        // the side whose pieces are hidden (0 = player +1), -1 for the state key; the viewer as sx_sample_hidden_states
        // reads it: viewer[b] == 1 is +1, anything else -1, NULL the player to move
        const int opp = !infoset ? -1 : viewer ? (viewer[b] == 1 ? 1 : 0) : a.to_move ^ 1;
        const uint8_t *gb = board + b * cfg.board_stride;
        int n = 0;
        for (int c0 = 0; c0 < cfg.N; c0 += 32) {
            const int c = c0 + lane;
            const uint32_t v = c < cfg.N ? gb[c] : 0u;
            const bool has = (v & CELL_RANK) != 0;  // the export writes nothing for a cell without a rank
            const uint32_t hb = __ballot_sync(FULL, has);
            if (has) occ[n + __popc(hb & lt)] = uint16_t(c | (v << 8));
            n += __popc(hb);
        }
        __syncwarp();

        const uint16_t *ce = cap + b * cfg.cap_stride;
        const int slots = 3 * n + KEY_EXTRA_SLOTS + a.ncap;
        uint64_t h = 0;
        for (int f = lane; f < slots; f += 32) {
            uint32_t c = 0, l, x;
            bool on = true;
            if (f < 3 * n) {
                const int seg = f < n ? 0 : f < 2 * n ? 1 : 2;
                const uint32_t e = occ[f - seg * n];
                const uint32_t v = e >> 8, rank = v & CELL_RANK, owner = (v >> 4) & 1;
                c = e & 255u;
                if (seg == 0) {  // true rank; a hidden cell shows its PO entry (UNKNOWN) in the information-set key
                    const bool hidden = int(owner) == opp && rank <= SP_BOMB && (v & (CELL_REVEALED | CELL_OBST)) == 0;
                    l = owner;
                    x = hidden ? SP_UNKNOWN : rank;
                } else if (seg == 1) {  // partially observable rank
                    l = 3 + owner;
                    x = (v & CELL_REVEALED) ? rank : SP_UNKNOWN;
                } else {  // never moved
                    l = 32 + owner;
                    x = 1;
                    on = (v & CELL_STILL) != 0;
                }
            } else if (f < 3 * n + KEY_EXTRA_SLOTS) {
                const int j = f - 3 * n;
                l = 5;
                switch (j) {  // the data layer: [0] turn, [1] over, [2] winner, [C] max_turns, [C + 1] invalid
                case 0: x = a.turn; break;
                case 1: c = 1; x = a.over; break;
                case 2: c = 2; x = a.winner; break;
                case 3: c = cfg.C; x = a.max_turns; break;
                case 4: c = cfg.C + 1; x = a.invalid; break;
                case 5: case 7: {  // recent moves of player +1 (layer 6) / -1 (layer 7): 1 on the from square
                    const int s = (j - 5) >> 1;
                    l = 6 + s;
                    c = a.rfrom[s];
                    x = 1;
                    on = c != NO_CELL;
                    break;
                }
                case 6: case 8: {  // -code on the to square
                    const int s = (j - 6) >> 1;
                    l = 6 + s;
                    c = a.rto[s];
                    x = uint32_t(-a.rcode[s]);
                    on = c != NO_CELL;
                    break;
                }
                case 9: l = KEY_LAYER_PLAYER; x = a.to_move == 0 ? 1u : uint32_t(-1); break;
                default: l = KEY_LAYER_VIEWER; x = opp == 1 ? 1u : uint32_t(-1); on = infoset != 0; break;
                }
            } else {  // capture entry: cell | owner << 8 | (type - 1) << 9 | (count - 1) << 13, one per (cell, owner, type)
                const uint32_t e = ce[f - 3 * n - KEY_EXTRA_SLOTS];
                c = e & 255u;
                l = 8 + 12 * ((e >> 8) & 1) + ((e >> 9) & 15);
                x = (e >> 13) + 1;
            }
            const uint64_t w = zobrist(c, l, x);
            if (on && x != 0) h ^= w;
        }
        const uint32_t lo = __reduce_xor_sync(FULL, uint32_t(h)), hi = __reduce_xor_sync(FULL, uint32_t(h >> 32));
        if (lane == 0) keys[b] = uint64_t(lo) | (uint64_t(hi) << 32);
        __syncwarp();  // the next game overwrites this one's cell list
    }
}

}  // namespace sx

extern "C" int sx_state_keys(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *viewer_d, uint32_t mode,
                             uint64_t *keys_d, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_state_keys: null config");
    if (null_state(st)) return sx_set_error("sx_state_keys: null state tensor");
    if (!keys_d) return sx_set_error("sx_state_keys: null keys");
    if (mode != SX_KEY_STATE && mode != SX_KEY_INFOSET)
        return sx_set_error("sx_state_keys: unknown mode " + std::to_string(mode));
    if (mode == SX_KEY_STATE && viewer_d) return sx_set_error("sx_state_keys: viewer_d must be NULL for SX_KEY_STATE");
    if (num_envs <= 0) return 0;
    const long long blocks = (num_envs + KEYS_WARPS - 1) / KEYS_WARPS;
    const unsigned grid = unsigned(blocks < 0x7fffffffLL ? blocks : 0x7fffffffLL);  // games beyond: the grid-stride loop
    sx_state_keys_kernel<<<grid, KEYS_WARPS * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        cfg->dev, st.board, st.aux, st.captured, num_envs, viewer_d, mode == SX_KEY_INFOSET ? 1 : 0, keys_d);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_state_keys_kernel", e);
}
