// sx_expand.cu -- the children of a node: every legal move of the player to move and the state it leads to.
//
// Search (PIMC, information-set MCTS, determinized rollouts) needs, per game, the list of moves of the player to move
// and the successor state of each.  Contract (include/stratego_b200.h, DESIGN.md §3.3):
//
//   children of game b: one per legal move of the player to move, identified by its flat spatial index in that player's
//   frame (the non-zero entries of the spatial mask without the noop channel A-1), in ascending index order.  A finished
//   game or a stuck player has none.  Child t of game b is row offsets[b] + t of the outputs and equals, byte for byte
//   (board with padding, aux, capture list, and the six scalars), what sx_step (spatial actions, no flags) makes of a
//   copy of game b with that action.
//
// Two launches.  sx_count_moves_kernel: one warp per game runs gen_moves for the player to move and sums the popcounts
// of the move sets.  sx_expand_moves_kernel: one warp per parent (grid-stride over the parents, so every warp takes
// dozens of them and a parent with a dozen scouts evens out against one with five moves) regenerates the move sets,
// numbers the moves in ascending flat-index order as sx_sample_policy_kernel does (running count per cell + binary
// search, 32 moves at a time, one per lane), writes the action list, and then plays the moves one after the other on a
// working copy of the parent staged in shared memory: apply_move, the next player's gen_moves, the outcome, the child row.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int EXPAND_WARPS = 8;  // warps per block of both kernels

template <int K, bool CM>
__global__ void __launch_bounds__(EXPAND_WARPS * 32) sx_count_moves_kernel(const __grid_constant__ DevConfig cfg,
                                                                           const uint8_t *board, const int16_t *aux,
                                                                           long long num_envs, int32_t *counts, int warp_bytes)
{
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * EXPAND_WARPS + warp;
    if (b >= num_envs) return;
    WarpMem m;
    carve_warp(cfg, smem + size_t(warp) * warp_bytes, &m);
    Aux a;
    unpack(load_game(cfg, board, aux, nullptr, b, m.board, nullptr), a);
    __syncwarp();
    gen_moves<K, Grp<1>, CM>(cfg, m, a, a.to_move, false);
    const int n = __reduce_add_sync(FULL, lane_moves<K>(cfg, m));
    if (lane == 0) counts[b] = n;
}

// one warp's shared memory beyond carve_warp: the parent's board and capture list, its move sets and the running move
// count per cell
__host__ __device__ inline int expand_warp_bytes(const DevConfig &cfg)
{
    return carve_warp(cfg, nullptr, nullptr) + round16(cfg.board_stride) + round16(cfg.cap_stride * 2) + round16(cfg.N * 8) +
           round16(cfg.N * 2);
}

template <int K, bool CM>
__global__ void __launch_bounds__(EXPAND_WARPS * 32, 3) sx_expand_moves_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap, long long num_envs,
    const int64_t *offsets, long long n_children, uint8_t *out_board, int16_t *out_aux, uint16_t *out_cap, int32_t *actions,
    sx_outputs o, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t *base = smem + size_t(warp) * warp_bytes;
    WarpMem m;
    int off = carve_warp(cfg, base, &m);
    uint8_t *pboard = base + off;
    off += round16(cfg.board_stride);
    uint16_t *pcap = reinterpret_cast<uint16_t *>(base + off);
    off += round16(cfg.cap_stride * 2);
    uint2 *pmoves = reinterpret_cast<uint2 *>(base + off);
    off += round16(cfg.N * 8);
    uint16_t *before = reinterpret_cast<uint16_t *>(base + off);  // [N] moves in the cells below p
    const int board_words = cfg.board_stride >> 2, cap_words = cfg.cap_stride >> 1;

    for (long long b = (long long)blockIdx.x * EXPAND_WARPS + warp; b < num_envs; b += (long long)gridDim.x * EXPAND_WARPS) {
        const long long start = offsets[b], end = offsets[b + 1];
        // offsets come from the caller and are not checked on the host: an empty slot or one that starts at or past
        // n_children writes nothing
        if (end <= start || start >= n_children) continue;
        const uint64_t slot = uint64_t(end) - uint64_t(start);
        const uint4 paw = load_game(cfg, board, aux, cap, b, pboard, pcap);
        for (int w = lane; w < board_words; w += 32) reinterpret_cast<uint32_t *>(m.board)[w] = reinterpret_cast<const uint32_t *>(pboard)[w];
        Aux pa;
        unpack(paw, pa);
        __syncwarp();
        gen_moves<K, GT, CM>(cfg, m, pa, pa.to_move, false);
        int mine, incl;
        const int total = lane_move_scan<K>(cfg, m, mine, incl);
        {
            int run = incl - mine;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const int p = lane * K + k;
                if (p < cfg.N) {
                    before[p] = uint16_t(run);
                    pmoves[p] = m.moves[p];
                    run += __popc(m.moves[p].x) + __popc(m.moves[p].y);
                }
            }
        }
        // children t in [first, lim) are written: t < the count, t < the slot, start + t in [0, n_children).  Both
        // differences are exact in uint64 (start < n_children, start < end), and lim <= total fits an int.
        const uint64_t room = uint64_t(n_children) - uint64_t(start);
        uint64_t lim64 = slot < room ? slot : room;
        lim64 = lim64 < uint64_t(total) ? lim64 : uint64_t(total);
        const int lim = int(lim64);
        const int first = start >= 0 ? 0 : start + lim <= 0 ? lim : int(-start);
        __syncwarp();
        const int mover = pa.to_move;
        for (int t0 = first; t0 < lim; t0 += 32) {
            // moves t0 .. t0 + 31: move t0 + lane is decoded by this lane (its cell by binary search in the running count)
            int my_action = 0;
            const int tl = t0 + lane;
            if (tl < lim) {
                int lo = 0, hi = cfg.N;
                while (hi - lo > 1) {
                    const int mid = (lo + hi) >> 1;
                    if (int(before[mid]) <= tl) lo = mid; else hi = mid;
                }
                my_action = lo * cfg.A + nth_set_bit64(pmoves[lo], tl - int(before[lo]));
                actions[start + tl] = my_action;
            }
            const int nb = lim - t0 < 32 ? lim - t0 : 32;
            for (int j = 0; j < nb; ++j) {
                const long long row = start + t0 + j;
                const int action = __shfl_sync(FULL, my_action, j);
                // the working copy of the parent
                for (int w = lane; w < board_words; w += 32)
                    reinterpret_cast<uint32_t *>(m.board)[w] = reinterpret_cast<const uint32_t *>(pboard)[w];
                for (int w = lane; w < cap_words; w += 32) reinterpret_cast<uint32_t *>(m.cap)[w] = reinterpret_cast<const uint32_t *>(pcap)[w];
                Aux a = pa;
                __syncwarp();
                // sx_step of the fused kernel (sx_kernels.cu, sx_fused_kernel: step, "move list of the player the outputs
                // are for", outcome, scalars, state write-back) for a spatial action without flags; kept in step with it
                // by tests/test_expand_moves_gpu.py, which compares every child with sx_step
                const Move mv = decode_spatial(cfg, action, mover);
                int attack;
                const StepStatus status = apply_move<GT>(cfg, m, a, mv, false, attack);
                if (status == STEP_MOVED) after_move<K, GT, CM>(cfg, m, a, mover);
                uint32_t w4[4];
                aux_pack(a, w4);
                if (status == STEP_ILLEGAL) {  // not reached for a generated move; sx_step leaves the state as it was
                    w4[0] = paw.x; w4[1] = paw.y; w4[2] = paw.z; w4[3] = paw.w;
                }
                // the child row, written here rather than with store_game / store_step_scalars (sx_device.cuh): with
                // those the expand pass took 0.8 % (Barrage) to 1.6 % (Standard) longer on a B200
                const bool done = status != STEP_ILLEGAL && a.over;
                uint32_t *ob = reinterpret_cast<uint32_t *>(out_board + row * cfg.board_stride);
                for (int w = lane; w < board_words; w += 32) ob[w] = reinterpret_cast<const uint32_t *>(m.board)[w];
                uint32_t *oc = reinterpret_cast<uint32_t *>(out_cap + row * cfg.cap_stride);
                for (int w = lane; w < cap_words; w += 32) oc[w] = reinterpret_cast<const uint32_t *>(m.cap)[w];
                if (lane == 0) {
                    *reinterpret_cast<uint4 *>(out_aux + row * 8) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
                    const int win = a.winner;
                    if (o.done) o.done[row] = done ? 1 : 0;
                    if (o.winner) o.winner[row] = int8_t(done ? win : 0);
                    if (o.ending_invalid) o.ending_invalid[row] = (done && a.invalid) ? 1 : 0;
                    if (o.illegal) o.illegal[row] = status == STEP_ILLEGAL ? 1 : (a.overflow ? 2 : 0);
                    if (o.reward) o.reward[row] = (done && !a.invalid) ? float(win) : 0.0f;  // maenv:777-801
                    if (o.player) o.player[row] = a.to_move == 0 ? 1 : -1;
                }
                __syncwarp();  // the next child's working copy overwrites what was just stored
            }
        }
        __syncwarp();  // the next parent overwrites this one's slices
    }
}

typedef void (*count_fn)(DevConfig, const uint8_t *, const int16_t *, long long, int32_t *, int);
typedef void (*expand_fn)(DevConfig, const uint8_t *, const int16_t *, const uint16_t *, long long, const int64_t *, long long,
                          uint8_t *, int16_t *, uint16_t *, int32_t *, sx_outputs, int);

}  // namespace sx

extern "C" int sx_count_moves(const sx_config *cfg, sx_state st, int64_t num_envs, int32_t *counts_d, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_count_moves: null config");
    if (null_state(st)) return sx_set_error("sx_count_moves: null state tensor");
    if (!counts_d) return sx_set_error("sx_count_moves: null counts");
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = carve_warp(d, nullptr, nullptr);
    const count_fn k = pick<count_fn>(cfg, sx_count_moves_kernel<2, false>, sx_count_moves_kernel<4, false>,
                                      sx_count_moves_kernel<4, true>, sx_count_moves_kernel<8, false>);
    const unsigned grid = unsigned((num_envs + EXPAND_WARPS - 1) / EXPAND_WARPS);
    k<<<grid, EXPAND_WARPS * 32, size_t(EXPAND_WARPS) * warp_bytes, static_cast<cudaStream_t>(stream)>>>(
        d, st.board, st.aux, num_envs, counts_d, warp_bytes);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_count_moves_kernel", e);
}

extern "C" int sx_expand_moves(const sx_config *cfg, sx_state st, int64_t num_envs, const int64_t *offsets_d,
                               int64_t n_children, sx_state out, int32_t *actions_d, sx_outputs out_scalars, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_expand_moves: null config");
    if (null_state(st)) return sx_set_error("sx_expand_moves: null state tensor");
    if (null_state(out)) return sx_set_error("sx_expand_moves: null out tensor");
    if (!actions_d) return sx_set_error("sx_expand_moves: null actions");
    if (!offsets_d) return sx_set_error("sx_expand_moves: null offsets");
    if (out.board == st.board)
        return sx_set_error("sx_expand_moves: out.board is st.board; the children need a state of their own");
    if (n_children < 0) return sx_set_error("sx_expand_moves: n_children must be >= 0, got " + std::to_string(n_children));
    const sx_outputs &o = out_scalars;
    if (!scalars_only(o)) return sx_set_error(std::string("sx_expand_moves") + NOT_SCALARS_ONLY);
    if (num_envs <= 0 || n_children == 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = expand_warp_bytes(d);
    const size_t smem = size_t(EXPAND_WARPS) * warp_bytes;
    const expand_fn k = pick<expand_fn>(cfg, sx_expand_moves_kernel<2, false>, sx_expand_moves_kernel<4, false>,
                                        sx_expand_moves_kernel<4, true>, sx_expand_moves_kernel<8, false>);
    // as many blocks as are resident at once: every warp loops over many parents, which evens out their move counts
    unsigned grid = 0;
    cudaError_t e = resident_grid(k, EXPAND_WARPS * 32, smem, (num_envs + EXPAND_WARPS - 1) / EXPAND_WARPS, grid);
    if (e != cudaSuccess) return fail("sx_expand_moves", e);
    k<<<grid, EXPAND_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(d, st.board, st.aux, st.captured, num_envs, offsets_d,
                                                                          n_children, out.board, out.aux, out.captured,
                                                                          actions_d, o, warp_bytes);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_expand_moves_kernel", e);
}
