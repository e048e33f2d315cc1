// sx_hidden.cu -- determinization: complete game states that agree with what one player knows.
//
// Stratego hides the opponent's pieces.  Search (PIMC, information-set MCTS, determinized rollouts) and belief-model
// training need whole game states that are consistent with one player's information instead of the TRUE state.  On a
// reachable state that information about an unrevealed enemy piece is (a) which of the enemy's unrevealed pieces are
// still on the board -- the multiset of their codes -- and (b) that a piece which has moved is neither a flag nor a bomb
// (a scout that moves more than one square is revealed, apply_move in sx_device.cuh).  This kernel draws placements of
// that multiset uniformly among those respecting (b).  Contract (include/stratego_b200.h, DESIGN.md §3.3):
//
//   hidden cells: cells holding a piece of the viewer's opponent that is not CELL_REVEALED, on no obstacle;
//   S = hidden cells with CELL_STILL, I = flags + bombs among their codes, M = the other codes.
//   Immovables: the still hidden cells ordered by (x, cell) ascending; rank j < I gets the j-th immovable code in
//   ascending order (flag before bombs).  Movables: every hidden cell not filled so ordered by (y, cell) ascending; rank
//   j gets the j-th movable code in ascending order.  x, y: the first two words of one Philox4x32-10 block per hidden
//   cell, key (seed lo, seed hi), counter (gid lo, gid hi, RNG_HIDDEN ^ draw, (sample << 8) | cell), gid = env_base + b.
//   Only the CELL_RANK nibble of hidden cells changes; I > S: the row is copied unchanged and status[b] = 1.
//
// One warp per OUTPUT row (game b, sample k): 64 games x 4 096 samples fill the GPU like 262 144 games x 1.  The warp
// stages the board row in shared memory, lists its hidden cells in ascending cell order (ballots), counts the codes
// (packed byte counters, one warp reduction per four codes), computes one Philox block per hidden cell (list entry i
// goes to lane i mod 32), and ranks each cell by counting the smaller (key, cell) pairs of the list in shared memory
// (every lane reads the same entry at the same time: a broadcast).  Any number of hidden cells up to the board's cells
// works, so custom boards with more than 40 pieces a side are covered.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int HIDDEN_WARPS = 8;  // warps per block
constexpr uint64_t NO_KEY = ~0ull;  // a list entry that does not take part in a ranking

// one warp's shared memory: the board row, the two key arrays (uint64 per hidden cell) and the hidden-cell list
// (cell | CELL_STILL-flag << 8 per entry, ascending cell order)
__host__ __device__ inline int hidden_warp_bytes(const DevConfig &cfg)
{
    return cfg.board_stride + 2 * round16(cfg.N * 8) + round16(cfg.N * 2);
}

// byte t & 3 of the packed code counters: the number of hidden cells holding code t + 1
__device__ __forceinline__ int code_count(uint32_t h0, uint32_t h1, uint32_t h2, int t)
{
    const uint32_t w = t < 4 ? h0 : t < 8 ? h1 : h2;
    return int((w >> (8 * (t & 3))) & 0xffu);
}

__global__ void __launch_bounds__(HIDDEN_WARPS * 32) sx_sample_hidden_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
    long long num_envs, long long env_base, const int8_t *viewer, int n_samples, uint2 key, uint32_t draw,
    uint8_t *out_board, int16_t *out_aux, uint16_t *out_cap, uint8_t *status, int warp_bytes)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *brd = smem + size_t(warp) * warp_bytes;
    uint64_t *kx = reinterpret_cast<uint64_t *>(brd + cfg.board_stride);
    uint64_t *ky = kx + round16(cfg.N * 8) / 8;
    uint16_t *cel = reinterpret_cast<uint16_t *>(ky + round16(cfg.N * 8) / 8);
    const uint32_t lt = (1u << lane) - 1u;
    const int board_words = cfg.board_stride >> 2, cap_vecs = cfg.cap_stride >> 3;  // cap_stride is a multiple of 8
    const long long rows = num_envs * n_samples;

    for (long long row = (long long)blockIdx.x * HIDDEN_WARPS + warp; row < rows; row += (long long)gridDim.x * HIDDEN_WARPS) {
        const long long b = row / n_samples;
        const uint32_t k = uint32_t(row - b * n_samples);
        const uint32_t *gb = reinterpret_cast<const uint32_t *>(board + b * cfg.board_stride);
        for (int w = lane; w < board_words; w += 32) reinterpret_cast<uint32_t *>(brd)[w] = gb[w];
        const uint4 aw = *reinterpret_cast<const uint4 *>(aux + b * 8);
        Aux a;
        {
            const uint32_t w[4] = {aw.x, aw.y, aw.z, aw.w};
            aux_unpack(w, a);
        }
        // the viewer's side (0 = player +1): viewer[b] == 1 is +1, anything else -1, as player_override of the step
        const int side = viewer ? (viewer[b] == 1 ? 0 : 1) : a.to_move;
        const int opp = side ^ 1;
        __syncwarp();

        // the hidden cells in ascending cell order, their still count and the counts of their codes
        int n = 0, S = 0;
        uint32_t h0 = 0, h1 = 0, h2 = 0;
        for (int c0 = 0; c0 < cfg.N; c0 += 32) {
            const int c = c0 + lane;
            const uint32_t v = c < cfg.N ? brd[c] : 0u;
            const int code = v & CELL_RANK;
            const bool hid = code != 0 && code <= SP_BOMB && int((v >> 4) & 1) == opp && (v & (CELL_REVEALED | CELL_OBST)) == 0;
            const bool still = hid && (v & CELL_STILL) != 0;
            const uint32_t hb = __ballot_sync(FULL, hid), sb = __ballot_sync(FULL, still);
            if (hid) {
                cel[n + __popc(hb & lt)] = uint16_t(c | (still ? 256 : 0));
                const int t = code - 1;
                const uint32_t inc = 1u << (8 * (t & 3));  // at most 8 cells per lane and 225 per warp: bytes never carry
                h0 += t < 4 ? inc : 0u;
                h1 += (t >= 4 && t < 8) ? inc : 0u;
                h2 += t >= 8 ? inc : 0u;
            }
            n += __popc(hb);
            S += __popc(sb);
        }
        h0 = __reduce_add_sync(FULL, h0);
        h1 = __reduce_add_sync(FULL, h1);
        h2 = __reduce_add_sync(FULL, h2);
        const int n_flag = code_count(h0, h1, h2, SP_FLAG - 1), I = n_flag + code_count(h0, h1, h2, SP_BOMB - 1);
        if (status && k == 0 && lane == 0) status[b] = I > S ? 1 : 0;
        __syncwarp();

        if (I <= S && n > 0) {  // warp-uniform; I > S: no placement exists, the row is copied unchanged
            const uint64_t gid = uint64_t(env_base + b);
            const uint32_t c2 = RNG_HIDDEN ^ draw;
            for (int i = lane; i < n; i += 32) {
                const uint32_t e = cel[i];
                const uint32_t c = e & 255u;
                const uint4 r = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), c2, (k << 8) | c), key);
                kx[i] = (e & 256u) ? ((uint64_t(r.x) << 8) | c) : NO_KEY;
                ky[i] = (uint64_t(r.y) << 8) | c;
            }
            __syncwarp();
            // immovables: the still cells of rank < I by (x, cell) get the flags, then the bombs; they leave the movables'
            // ranking (their y key becomes NO_KEY, written by the entry's own lane: nobody reads ky here)
            if (I > 0) {
                for (int i0 = 0; i0 < n; i0 += 32) {
                    const int i = i0 + lane;
                    const uint64_t mine = i < n ? kx[i] : NO_KEY;
                    int r = 0;
                    for (int e = 0; e < n; ++e) r += kx[e] < mine ? 1 : 0;
                    if (mine != NO_KEY && r < I) {
                        const int c = cel[i] & 255;
                        brd[c] = uint8_t((brd[c] & ~CELL_RANK) | uint32_t(r < n_flag ? SP_FLAG : SP_BOMB));
                        ky[i] = NO_KEY;
                    }
                }
                __syncwarp();
            }
            // movables: every other hidden cell by (y, cell); rank r gets the r-th movable code in ascending order,
            // 1 + the number of codes t whose running count through t is <= r
            for (int i0 = 0; i0 < n; i0 += 32) {
                const int i = i0 + lane;
                const uint64_t mine = i < n ? ky[i] : NO_KEY;
                int r = 0;
                for (int e = 0; e < n; ++e) r += ky[e] < mine ? 1 : 0;
                if (mine != NO_KEY) {
                    int code = 1, cum = 0;
#pragma unroll
                    for (int t = 0; t < SP_MARSHAL; ++t) {
                        cum += code_count(h0, h1, h2, t);
                        code += cum <= r ? 1 : 0;
                    }
                    const int c = cel[i] & 255;
                    brd[c] = uint8_t((brd[c] & ~CELL_RANK) | uint32_t(code));
                }
            }
            __syncwarp();
        }

        uint32_t *ob = reinterpret_cast<uint32_t *>(out_board + row * cfg.board_stride);
        for (int w = lane; w < board_words; w += 32) ob[w] = reinterpret_cast<const uint32_t *>(brd)[w];
        if (lane == 0) *reinterpret_cast<uint4 *>(out_aux + row * 8) = aw;
        const uint4 *gc = reinterpret_cast<const uint4 *>(cap + b * cfg.cap_stride);
        uint4 *oc = reinterpret_cast<uint4 *>(out_cap + row * cfg.cap_stride);
        for (int w = lane; w < cap_vecs; w += 32) oc[w] = gc[w];
        __syncwarp();  // the next row's loads overwrite this warp's shared memory
    }
}

}  // namespace sx

extern "C" int sx_sample_hidden_states(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base,
                                       const int8_t *viewer_d, int32_t n_samples, uint64_t seed, uint32_t draw,
                                       sx_state out, uint8_t *status_d, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_sample_hidden_states: null config");
    if (null_state(st)) return sx_set_error("sx_sample_hidden_states: null state tensor");
    if (null_state(out)) return sx_set_error("sx_sample_hidden_states: null out tensor");
    if (n_samples < 1 || n_samples >= (1 << 24))
        return sx_set_error("sx_sample_hidden_states: n_samples must be in [1, 2^24), got " + std::to_string(n_samples));
    // rows * board_stride (<= 240 bytes) must stay a valid int64 byte offset
    if (num_envs > 0 && num_envs > (INT64_MAX >> 8) / n_samples)
        return sx_set_error("sx_sample_hidden_states: num_envs * n_samples overflows the row count (num_envs " +
                            std::to_string(num_envs) + ", n_samples " + std::to_string(n_samples) + ")");
    if (out.board == st.board)
        return sx_set_error("sx_sample_hidden_states: out.board is st.board; the samples need a state of their own");
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = hidden_warp_bytes(d);
    const long long rows = (long long)num_envs * n_samples;
    const long long blocks = (rows + HIDDEN_WARPS - 1) / HIDDEN_WARPS;
    const unsigned grid = unsigned(blocks < 0x7fffffffLL ? blocks : 0x7fffffffLL);  // rows beyond: the grid-stride loop
    const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
    sx_sample_hidden_kernel<<<grid, HIDDEN_WARPS * 32, size_t(HIDDEN_WARPS) * warp_bytes, static_cast<cudaStream_t>(stream)>>>(
        d, st.board, st.aux, st.captured, num_envs, env_base, viewer_d, n_samples, key, draw, out.board, out.aux,
        out.captured, status_d, warp_bytes);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_sample_hidden_kernel", e);
}
