// sx_playout.cu -- play games out on the device: uniformly random legal moves until the game ends or a ply cap.
//
// Search scores a leaf by playing it out.  Contract (include/stratego_b200.h, DESIGN.md §3.3): the move of every ply is
// the fused step's SX_SAMPLE_NEXT draw for the state before that ply (Philox4x32-10, key (seed lo, seed hi), counter
// (gid lo, gid hi, RNG_SAMPLE ^ turn, episode), gid = env_base + b, first word, sample_move), so a playout of n plies
// equals, byte for byte, a chain of n fused steps (spatial actions, SX_SAMPLE_NEXT, no auto-reset, same seed and
// env_base) that stops at the first step reporting done.  A player to move without a move (only an imported state can
// be so) plays the noop and loses, as a step with the 1D noop action does.  A game over at entry plays nothing.
//
// One warp per game, Grp<1> on every board (a ≤ 16-cell board leaves most lanes idle, as in sx_expand.cu).  The game's
// board and capture list stay in the warp's shared slice and its aux in registers from the load to the write-back; per
// ply: the draw over the move sets, decode_spatial, apply_move and after_move, whose move sets of the next player feed
// the next draw (one move generation per ply).  Random games differ a lot in length, so warps claim games dynamically:
// the grid holds only the resident blocks, block k owns a contiguous range of games, and its warps take the next game
// of the range from a shared-memory counter.
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int PLAYOUT_WARPS = 8;  // warps per block

template <int K, bool CM>
__global__ void __launch_bounds__(PLAYOUT_WARPS * 32, 4) sx_playout_kernel(
    const __grid_constant__ DevConfig cfg, uint8_t *board, int16_t *aux, uint16_t *cap, long long num_envs,
    long long env_base, long long per_block, int max_plies, uint2 key, int32_t *plies_out, sx_outputs o, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ unsigned long long claimed;  // games of this block's range handed out so far
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) claimed = 0;
    __syncthreads();
    WarpMem m;
    carve_warp(cfg, smem + size_t(warp) * warp_bytes, &m);
    for (long long b; (b = claim_next(claimed, per_block, num_envs)) >= 0;) {
        Aux a;
        unpack(load_game(cfg, board, aux, cap, b, m.board, m.cap), a);
        __syncwarp();
        const uint64_t gid = uint64_t(env_base + b);
        int plies = 0;
        if (!a.over && max_plies > 0) {
            bool any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);
            for (;;) {
                const int mover = a.to_move;
                int attack;
                ++plies;
                if (!any) {  // impl:809-814, 912-920: the stuck player's noop loses (the draw is the noop entry A-1)
                    apply_move<GT>(cfg, m, a, Move{0, 0, 0, 0, 0, 0, true, false}, false, attack);
                    break;
                }
                // the draw sx_fused_kernel makes for SX_SAMPLE_NEXT on this state (sx_kernels.cu)
                const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SAMPLE ^ uint32_t(a.turn), a.episode), key);
                const int action = sample_move<K, GT>(cfg, m, true, rnd.x);
                apply_move<GT>(cfg, m, a, decode_spatial(cfg, action, mover), false, attack);
                any = after_move<K, GT, CM>(cfg, m, a, mover);
                if (a.over || plies >= max_plies) break;
            }
            uint32_t w4[4];
            aux_pack(a, w4);
            store_game(cfg, m, w4, board, aux, cap, b);
        }
        if (lane == 0) {  // the scalars of the step that ended the game
            if (plies_out) plies_out[b] = plies;
            store_step_scalars(o, b, a, a.over, a.overflow ? 2 : 0);
        }
        __syncwarp();  // the next game overwrites this one's slice
    }
}

typedef void (*playout_fn)(DevConfig, uint8_t *, int16_t *, uint16_t *, long long, long long, long long, int, uint2,
                           int32_t *, sx_outputs, int);

}  // namespace sx

extern "C" int sx_playout(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, int32_t max_plies,
                          uint64_t seed, int32_t *plies_d, sx_outputs out_scalars, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_playout: null config");
    if (null_state(st)) return sx_set_error("sx_playout: null state tensor");
    if (max_plies < 0) return sx_set_error("sx_playout: max_plies must be >= 0, got " + std::to_string(max_plies));
    const sx_outputs &o = out_scalars;
    if (!scalars_only(o)) return sx_set_error(std::string("sx_playout") + NOT_SCALARS_ONLY);
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = carve_warp(d, nullptr, nullptr);
    const size_t smem = size_t(PLAYOUT_WARPS) * warp_bytes;
    const playout_fn k = pick<playout_fn>(cfg, sx_playout_kernel<2, false>, sx_playout_kernel<4, false>,
                                          sx_playout_kernel<4, true>, sx_playout_kernel<8, false>);
    unsigned grid = 0;
    long long per_block = 0;
    cudaError_t e = claim_grid(k, PLAYOUT_WARPS, smem, num_envs, grid, per_block);
    if (e != cudaSuccess) return fail("sx_playout", e);
    const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
    k<<<grid, PLAYOUT_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(d, st.board, st.aux, st.captured, num_envs,
                                                                           env_base, per_block, max_plies, key, plies_d, o,
                                                                           warp_bytes);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_playout_kernel", e);
}
