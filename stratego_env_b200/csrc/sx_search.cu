// sx_search.cu -- Monte Carlo tree search on the device: a fixed number of iterations per root, one launch, one warp
// per tree.
//
// Contract (include/stratego_b200.h, DESIGN.md §3.3): game b is the root (node 0) of its own tree of at most max_nodes
// nodes, stored struct-of-arrays [B, max_nodes].  Iteration i: descend from the root, taking the first unvisited child
// or else the child of best PUCT score (uniform prior, float32 without contraction, ties to the lowest index); a leaf
// that is not over gets all its children, in ascending flat spatial index (the expand_moves action list), when the pool
// has room for them; stop at the first child visited for the first time, at a finished state or at a leaf.  Evaluate
// the state reached: the winner if it is over, else a random playout of at most max_plies plies with the search's draw
// (counter (gid lo, gid hi, RNG_SEARCH ^ i, turn), sample_move numbering, a stuck player plays the noop and loses).
// Back the result up the path: N += 1, W += z.
//
// One warp per tree, with sx_playout's launch shape: the grid holds only the resident blocks, block k owns a
// contiguous range of trees, and its warps take the next tree of the range from a shared-memory counter.  The state of
// the current iteration lives in the warp's shared slice (board, capture list; aux in registers) and is rebuilt from
// the root each iteration by replaying the stored actions of the path (decode_spatial, apply_move, after_move); the
// tree lives in global memory, where a selection pass reads 32 children's N and W coalesced, one per lane, and takes a
// warp argmax by (score, index).
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int SEARCH_WARPS = 8;  // warps per block

template <int K, bool CM>
__global__ void __launch_bounds__(SEARCH_WARPS * 32, 4) sx_search_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
    long long num_envs, long long env_base, long long per_block, int iterations, int max_nodes, int max_plies,
    float c_explore, uint2 key, sx_tree tree, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ unsigned long long claimed;  // trees of this block's range handed out so far
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) claimed = 0;
    __syncthreads();
    WarpMem m;
    carve_warp(cfg, smem + size_t(warp) * warp_bytes, &m);
    for (long long b; (b = claim_next(claimed, per_block, num_envs)) >= 0;) {
        const uint64_t gid = uint64_t(env_base + b);
        const long long row = b * (long long)max_nodes;
        int32_t *const N = tree.visits + row, *const W = tree.value + row, *const parent = tree.parent + row;
        int32_t *const first_child = tree.first_child + row, *const n_children = tree.n_children + row;
        int32_t *const action = tree.action + row;
        if (lane == 0) { N[0] = 0; W[0] = 0; parent[0] = -1; first_child[0] = -1; n_children[0] = 0; action[0] = -1; }
        int used = 1;
        for (int it = 0; it < iterations; ++it) {
            Aux a;
            unpack(load_game(cfg, board, aux, cap, b, m.board, m.cap), a);
            __syncwarp();  // also orders the previous iteration's tree stores of lane 0 before this iteration's loads
            // ---- descent: v and the state after its path; `fresh`: m.moves holds the moves of the state's player
            int v = 0;
            bool fresh = false, any = false;
            for (;;) {
                if (a.over) break;
                int f = first_child[v], n = n_children[v];
                if (f < 0) {
                    if (!fresh) { any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false); fresh = true; }
                    int mine, incl;
                    n = lane_move_scan<K>(cfg, m, mine, incl);
                    if (n == 0 || n > max_nodes - used) break;  // a stuck player, or no room: v stays a leaf
                    f = used;
                    int t = f + incl - mine;  // this lane's children
                    for_each_lane_move<K>(cfg, m, [&](int act) {
                        const int c = t++;
                        N[c] = 0; W[c] = 0; parent[c] = v; first_child[c] = -1; n_children[c] = 0; action[c] = act;
                    });
                    if (lane == 0) { first_child[v] = f; n_children[v] = n; }
                    used += n;
                    __syncwarp();  // the children's fields, written by their lanes, are read below by others
                }
                // ---- selection: the first child with N = 0, else the argmax of q + u (lowest index on a tie)
                const float sqrt_nv = __fsqrt_rn(float(N[v]));
                const int sigma = a.to_move == 0 ? 1 : -1;
                float best = 0.0f;
                int best_j = -1, fresh_child = -1;
                for (int j0 = 0; j0 < n; j0 += 32) {
                    const int j = j0 + lane;
                    int nc = 1, wc = 0;
                    if (j < n) { nc = N[f + j]; wc = W[f + j]; }
                    const uint32_t zero = __ballot_sync(FULL, nc == 0);
                    if (zero) { fresh_child = j0 + __ffs(zero) - 1; break; }
                    if (j < n) {
                        const float q = __fdiv_rn(float(sigma * wc), float(nc));
                        const float u = __fdiv_rn(__fmul_rn(c_explore, sqrt_nv), float(1 + nc));
                        const float s = __fadd_rn(q, u);
                        if (best_j < 0 || s > best) { best = s; best_j = j; }  // j ascends: ties keep the lower index
                    }
                }
                int c;
                if (fresh_child >= 0) {
                    c = fresh_child;
                } else {
                    warp_argmax(best, best_j);
                    c = best_j;
                }
                // ---- step to the child: what expand_moves / sx_step make of s with that action
                const int mover = a.to_move;
                int attack;
                apply_move<GT>(cfg, m, a, decode_spatial(cfg, action[f + c], mover), false, attack);
                any = after_move<K, GT, CM>(cfg, m, a, mover);
                fresh = true;
                v = f + c;
                if (fresh_child >= 0) break;
            }
            // ---- evaluation: player +1's reward of the state reached, or of a random playout from it
            if (!a.over && max_plies > 0) {
                if (!fresh) any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);
                for (int plies = 1;; ++plies) {
                    const int mover = a.to_move;
                    int attack;
                    if (!any) {  // impl:809-814, 912-920: the stuck player's noop loses
                        apply_move<GT>(cfg, m, a, Move{0, 0, 0, 0, 0, 0, true, false}, false, attack);
                        break;
                    }
                    const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SEARCH ^ uint32_t(it),
                                                               uint32_t(a.turn) & 0xffffu), key);
                    const int act = sample_move<K, GT>(cfg, m, true, rnd.x);
                    apply_move<GT>(cfg, m, a, decode_spatial(cfg, act, mover), false, attack);
                    any = after_move<K, GT, CM>(cfg, m, a, mover);
                    if (a.over || plies >= max_plies) break;
                }
            }
            const int z = a.over && !a.invalid ? a.winner : 0;
            // ---- backup: the path is v and its ancestors
            if (lane == 0) {
                for (int x = v; x >= 0; x = parent[x]) { N[x] += 1; W[x] += z; }
            }
            __syncwarp();  // the next iteration's state overwrites this one's slice
        }
        if (lane == 0) tree.used[b] = used;
    }
}

typedef void (*search_fn)(DevConfig, const uint8_t *, const int16_t *, const uint16_t *, long long, long long, long long,
                          int, int, int, float, uint2, sx_tree, int);

}  // namespace sx

extern "C" int sx_search(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, int32_t iterations,
                         int32_t max_nodes, int32_t max_plies, float c_explore, uint64_t seed, sx_tree tree, void *stream)
{
    using namespace sx;
    if (!cfg) return sx_set_error("sx_search: null config");
    if (null_state(st)) return sx_set_error("sx_search: null state tensor");
    if (!tree.visits || !tree.value || !tree.parent || !tree.first_child || !tree.n_children || !tree.action || !tree.used)
        return sx_set_error("sx_search: null tree pointer");
    if (iterations < 0 || iterations > (1 << 24))
        return sx_set_error("sx_search: iterations must be in [0, 2^24], got " + std::to_string(iterations));
    if (max_nodes < 1) return sx_set_error("sx_search: max_nodes must be >= 1, got " + std::to_string(max_nodes));
    if (max_plies < 0) return sx_set_error("sx_search: max_plies must be >= 0, got " + std::to_string(max_plies));
    if (!(c_explore >= 0.0f) || c_explore > 3.4028235e38f)  // NaN fails the first test, +inf the second
        return sx_set_error("sx_search: c_explore must be finite and >= 0, got " + std::to_string(c_explore));
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = carve_warp(d, nullptr, nullptr);
    const size_t smem = size_t(SEARCH_WARPS) * warp_bytes;
    const search_fn k = pick<search_fn>(cfg, sx_search_kernel<2, false>, sx_search_kernel<4, false>,
                                        sx_search_kernel<4, true>, sx_search_kernel<8, false>);
    unsigned grid = 0;
    long long per_block = 0;
    cudaError_t e = claim_grid(k, SEARCH_WARPS, smem, num_envs, grid, per_block);
    if (e != cudaSuccess) return fail("sx_search", e);
    const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
    k<<<grid, SEARCH_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(d, st.board, st.aux, st.captured, num_envs,
                                                                          env_base, per_block, iterations, max_nodes,
                                                                          max_plies, c_explore, key, tree, warp_bytes);
    e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_search_kernel", e);
}
