// sx_guided.cu -- tree search whose leaves the caller evaluates: PUCT selection and backup on the device, one launch
// each, one warp per tree.
//
// Contract (include/stratego_b200.h, DESIGN.md §3.3): game b is the root (node 0) of its own tree of at most max_nodes
// nodes, stored struct-of-arrays [B, max_nodes] like sx_search's, with a float32 value W and a float32 prior P.  A round
// is sx_guided_select (descend from the root by the PUCT score q + c_puct * P * sqrt(N_parent) / (1 + N), float32
// without contraction, ties to the lowest index, to the first node without children or whose state is over; write that
// leaf's state, node and kind), the caller's network on the leaf states, and sx_guided_backup (give an evaluable leaf
// without children its legal moves as children, with the softmax of the caller's logits over those moves as priors,
// when the pool has room; add the value to N and W of the leaf and its ancestors).
//
// One warp per tree, one tree per warp of the grid: a round is a short replay (a few plies) per tree, so the work per
// warp is even and sx_search's dynamic claiming buys nothing.  Select keeps the state in the warp's shared slice
// (carve_warp) and replays the stored path (decode_spatial, apply_move, after_move); the tree lives in global memory,
// where a selection pass reads 32 children's N, W and P coalesced, one per lane, and takes a warp argmax by (score,
// index).  Backup regenerates the leaf's moves from its state row (gen_moves), gathers each lane's logits at
// p * A + channel, and forms the softmax with a warp max, expf, a warp sum and a correctly rounded division; the children
// are written at each lane's prefix-sum offset, and lane 0 walks the parent links.
//
// Several leaves per tree (sx_guided_select_many / sx_guided_backup_many): the same two kernels take L.  Select loops
// over the L leaves inside the warp, each a replay from the root; after leaf j, lane 0 adds a pending visit along its
// path in the per-node int32 buffer `inflight`, which the next descents read next to N, W and P (the virtual-loss
// score), and before the warp ends it walks the L - 1 paths again and takes the visits back, so the buffer is zero
// before and after every call.  Leaf 0 never reads the buffer and V = 0 leaves the score unchanged, so L = 1 is the
// one-leaf select.  Backup takes the L leaves of its tree in order with the one-leaf code, so a node reached twice is
// expanded by the first leaf.  One code path for every L: at L = 1 it is no slower than the one-leaf kernels were
// (DESIGN.md §3.3), so there is no separate L = 1 instantiation.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

constexpr int GUIDED_WARPS = 8;  // warps per block

// logit i of a row in the caller's dtype (SX_DTYPE_*; checked on the host)
__device__ __forceinline__ float guided_logit(const void *row, int dtype, int i)
{
    if (dtype == SX_DTYPE_BF16) return __bfloat162float(static_cast<const __nv_bfloat16 *>(row)[i]);
    if (dtype == SX_DTYPE_F16) return __half2float(static_cast<const __half *>(row)[i]);
    return static_cast<const float *>(row)[i];
}

template <int K, bool CM>
__global__ void __launch_bounds__(GUIDED_WARPS * 32, 4) sx_guided_select_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
    long long num_envs, int max_nodes, float c_puct, float fpu, int L, float vl, int32_t *inflight, sx_guided_tree tree,
    uint8_t *leaf_board, int16_t *leaf_aux, uint16_t *leaf_cap, int32_t *leaf_node, int8_t *leaf_kind, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * GUIDED_WARPS + warp;
    if (b >= num_envs) return;
    WarpMem m;
    carve_warp(cfg, smem + size_t(warp) * warp_bytes, &m);
    const long long row = b * (long long)max_nodes;
    const int32_t *const N = tree.visits + row, *const first_child = tree.first_child + row;
    const int32_t *const n_children = tree.n_children + row, *const action = tree.action + row;
    const int32_t *const parent = tree.parent + row;
    const float *const W = tree.value + row, *const P = tree.prior + row;
    int32_t *const V = inflight + row;  // pending visits of this round's earlier leaves; read from leaf 1 on
#pragma unroll 1
    for (int j = 0; j < L; ++j) {
        const long long r = b * L + j;  // the leaf's output row
        const bool pend = j > 0;        // pending visits exist from leaf 1 on
        Aux a;
        unpack(load_game(cfg, board, aux, cap, b, m.board, m.cap), a);
        __syncwarp();
        // ---- descent: v and the state after its path; `fresh`: m.moves holds the moves of the state's player to move
        int v = 0;
        bool fresh = false, any = false;
        for (;;) {
            if (a.over) break;
            const int f = first_child[v], n = n_children[v];
            if (f < 0 || n <= 0) break;
            // the argmax of q + u over the children, 32 per pass (lowest index on a tie); with V = 0 (leaf 0, and
            // nodes off the earlier paths) vl * 0 = +0 and sigma * W - (+0) = sigma * W, so this is the one-leaf score
            const float sqrt_nv = __fsqrt_rn(float(N[v] + (pend ? V[v] : 0)));
            const bool plus = a.to_move == 0;
            float best = 0.0f;
            int best_j = -1;
            for (int c0 = 0; c0 < n; c0 += 32) {
                const int c = c0 + lane;
                if (c < n) {
                    const int vc = pend ? V[f + c] : 0, nc = N[f + c] + vc;
                    const float wc = W[f + c], pc = P[f + c];
                    const float sw = __fsub_rn(plus ? wc : -wc, __fmul_rn(vl, float(vc)));  // sigma W - vl V
                    const float q = nc > 0 ? __fdiv_rn(sw, float(nc)) : fpu;
                    const float u = __fdiv_rn(__fmul_rn(__fmul_rn(c_puct, pc), sqrt_nv), float(1 + nc));
                    const float s = __fadd_rn(q, u);
                    if (best_j < 0 || s > best) { best = s; best_j = c; }  // c ascends: ties keep the lower index
                }
            }
            warp_argmax(best, best_j);
            // ---- step to the child: what expand_moves / sx_step make of the state with that action
            const int mover = a.to_move;
            int attack;
            apply_move<GT>(cfg, m, a, decode_spatial(cfg, action[f + best_j], mover), false, attack);
            any = after_move<K, GT, CM>(cfg, m, a, mover);
            fresh = true;
            v = f + best_j;
        }
        if (!a.over && !fresh) any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);
        __syncwarp();
        // ---- the leaf's state row
        uint32_t w4[4];
        aux_pack(a, w4);
        store_game(cfg, m, w4, leaf_board, leaf_aux, leaf_cap, r);
        if (lane == 0) {
            leaf_node[r] = v;
            leaf_kind[r] = int8_t(a.over ? SX_LEAF_OVER : any ? SX_LEAF_EVAL : SX_LEAF_STUCK);
            if (j < L - 1)  // a pending visit on the path, for the leaves after this one
                for (int x = v; x >= 0; x = parent[x]) V[x] += 1;
        }
        __syncwarp();  // the pending visits and the shared slice are the whole warp's before the next descent
    }
    // ---- take the pending visits back: the buffer is all zero again
    if (lane == 0)
        for (int j = 0; j < L - 1; ++j)
            for (int x = leaf_node[b * L + j]; x >= 0; x = parent[x]) V[x] -= 1;
}

template <int K, bool CM>
__global__ void __launch_bounds__(GUIDED_WARPS * 32, 4) sx_guided_backup_kernel(
    const __grid_constant__ DevConfig cfg, const uint8_t *leaf_board, const int16_t *leaf_aux, const uint16_t *leaf_cap,
    long long num_envs, int max_nodes, int L, sx_guided_tree tree, const int32_t *leaf_node, const int8_t *leaf_kind,
    const uint8_t *logits, int dtype, int logit_bytes, const float *values, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long b = (long long)blockIdx.x * GUIDED_WARPS + warp;
    if (b >= num_envs) return;
    const long long row = b * (long long)max_nodes;
    int32_t *const N = tree.visits + row, *const parent = tree.parent + row, *const first_child = tree.first_child + row;
    int32_t *const n_children = tree.n_children + row, *const action = tree.action + row;
    float *const W = tree.value + row, *const P = tree.prior + row;
    int used = tree.used[b];
    // the leaves in order: leaf j sees the expansions of leaves 0 .. j-1, so a node reached by several is expanded once
#pragma unroll 1
    for (int j = 0; j < L; ++j) {
        const long long r = b * L + j;  // the leaf's row
        const int v = leaf_node[r], kind = leaf_kind[r];
        Aux a;
        unpack(*reinterpret_cast<const uint4 *>(leaf_aux + r * 8), a);
        // z: the value backed up, in absolute terms (+1 = player +1 wins)
        const float z = kind == SX_LEAF_EVAL ? (a.to_move == 0 ? values[r] : -values[r])
                      : kind == SX_LEAF_OVER ? float(a.over && !a.invalid ? a.winner : 0)
                                             : (a.to_move == 0 ? -1.0f : 1.0f);  // STUCK: the player to move loses
        int f = -1, n = 0;
        if (kind == SX_LEAF_EVAL && first_child[v] < 0) {
            WarpMem m;
            carve_warp(cfg, smem + size_t(warp) * warp_bytes, &m);
            load_game(cfg, leaf_board, leaf_aux, leaf_cap, r, m.board, m.cap);
            __syncwarp();
            gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);
            int mine, incl;
            const int total = lane_move_scan<K>(cfg, m, mine, incl);
            if (total > 0 && total <= max_nodes - used) {
                f = used;
                n = total;
                const uint8_t *lrow = logits + r * (long long)(cfg.N * cfg.A) * logit_bytes;
                // softmax over the legal entries: max, then sum of expf(x - max), both reduced over the warp
                float mx = -INFINITY;
                for_each_lane_move<K>(cfg, m, [&](int act) { mx = fmaxf(mx, guided_logit(lrow, dtype, act)); });
#pragma unroll
                for (int d = 16; d >= 1; d >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, d));
                const bool uniform = !(mx > -INFINITY);  // every legal logit is -inf: each child gets 1 / n
                float sum = 0.0f;
                if (!uniform) {
                    for_each_lane_move<K>(cfg, m, [&](int act) {
                        sum = __fadd_rn(sum, expf(__fsub_rn(guided_logit(lrow, dtype, act), mx)));
                    });
#pragma unroll
                    for (int d = 16; d >= 1; d >>= 1) sum = __fadd_rn(sum, __shfl_xor_sync(FULL, sum, d));  // same on every lane
                }
                int t = f + incl - mine;  // this lane's children
                for_each_lane_move<K>(cfg, m, [&](int act) {
                    const int c = t++;
                    N[c] = 0; W[c] = 0.0f; parent[c] = v; first_child[c] = -1; n_children[c] = 0; action[c] = act;
                    P[c] = uniform ? __fdiv_rn(1.0f, float(n))
                                   : __fdiv_rn(expf(__fsub_rn(guided_logit(lrow, dtype, act), mx)), sum);
                });
            }
        }
        // ---- backup: the leaf and its ancestors
        if (lane == 0) {
            if (n > 0) { first_child[v] = f; n_children[v] = n; }
            for (int x = v; x >= 0; x = parent[x]) { N[x] += 1; W[x] = __fadd_rn(W[x], z); }
        }
        used += n;
        __syncwarp();  // lane 0's links are the whole warp's before the next leaf reads them
    }
    if (lane == 0 && used != tree.used[b]) tree.used[b] = used;
}

typedef void (*guided_select_fn)(DevConfig, const uint8_t *, const int16_t *, const uint16_t *, long long, int, float,
                                 float, int, float, int32_t *, sx_guided_tree, uint8_t *, int16_t *, uint16_t *, int32_t *,
                                 int8_t *, int);
typedef void (*guided_backup_fn)(DevConfig, const uint8_t *, const int16_t *, const uint16_t *, long long, int, int,
                                 sx_guided_tree, const int32_t *, const int8_t *, const uint8_t *, int, int, const float *,
                                 int);

static bool null_tree(const sx_guided_tree &t)
{
    return !t.visits || !t.value || !t.parent || !t.first_child || !t.n_children || !t.action || !t.prior || !t.used;
}

static std::string fn_error(const char *fn, const std::string &what) { return std::string(fn) + ": " + what; }

static int guided_select(const char *fn, const sx_config *cfg, sx_state st, int64_t num_envs, sx_guided_tree tree,
                         int32_t max_nodes, float c_puct, float fpu, int32_t L, float vl, int32_t *inflight_d,
                         sx_state leaf_states, int32_t *leaf_node_d, int8_t *leaf_kind_d, void *stream)
{
    if (!cfg) return sx_set_error(fn_error(fn, "null config"));
    if (null_state(st)) return sx_set_error(fn_error(fn, "null state tensor"));
    if (null_tree(tree)) return sx_set_error(fn_error(fn, "null tree pointer"));
    if (null_state(leaf_states) || !leaf_node_d || !leaf_kind_d) return sx_set_error(fn_error(fn, "null leaf output"));
    if (leaf_states.board == st.board) return sx_set_error(fn_error(fn, "leaf_states.board is st.board"));
    if (max_nodes < 1) return sx_set_error(fn_error(fn, "max_nodes must be >= 1, got " + std::to_string(max_nodes)));
    if (!(c_puct >= 0.0f) || c_puct > 3.4028235e38f)  // NaN fails the first test, +inf the second
        return sx_set_error(fn_error(fn, "c_puct must be finite and >= 0, got " + std::to_string(c_puct)));
    if (!(fpu >= -3.4028235e38f && fpu <= 3.4028235e38f))
        return sx_set_error(fn_error(fn, "fpu must be finite, got " + std::to_string(fpu)));
    if (L < 1 || L > SX_GUIDED_MAX_LEAVES)
        return sx_set_error(fn_error(fn, "leaves_per_tree must be in [1, 1024], got " + std::to_string(L)));
    if (!(vl >= 0.0f && vl <= 16777216.0f))  // NaN fails both
        return sx_set_error(fn_error(fn, "virtual_loss must be in [0, 2^24], got " + std::to_string(vl)));
    if (L > 1 && !inflight_d) return sx_set_error(fn_error(fn, "null inflight buffer with leaves_per_tree > 1"));
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = carve_warp(d, nullptr, nullptr);
    const size_t smem = size_t(GUIDED_WARPS) * warp_bytes;
    const guided_select_fn k = pick<guided_select_fn>(cfg, sx_guided_select_kernel<2, false>,
                                                      sx_guided_select_kernel<4, false>, sx_guided_select_kernel<4, true>,
                                                      sx_guided_select_kernel<8, false>);
    const unsigned grid = unsigned((num_envs + GUIDED_WARPS - 1) / GUIDED_WARPS);
    k<<<grid, GUIDED_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        d, st.board, st.aux, st.captured, num_envs, max_nodes, c_puct, fpu, L, vl, inflight_d, tree, leaf_states.board,
        leaf_states.aux, leaf_states.captured, leaf_node_d, leaf_kind_d, warp_bytes);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_guided_select_kernel", e);
}

static int guided_backup(const char *fn, const sx_config *cfg, sx_state leaf_states, int64_t num_envs,
                         sx_guided_tree tree, int32_t max_nodes, int32_t L, const int32_t *leaf_node_d,
                         const int8_t *leaf_kind_d, const void *logits_d, int32_t logits_dtype, const float *values_d,
                         void *stream)
{
    if (!cfg) return sx_set_error(fn_error(fn, "null config"));
    if (null_state(leaf_states)) return sx_set_error(fn_error(fn, "null leaf state tensor"));
    if (null_tree(tree)) return sx_set_error(fn_error(fn, "null tree pointer"));
    if (!leaf_node_d || !leaf_kind_d) return sx_set_error(fn_error(fn, "null leaf node or kind"));
    if (!logits_d) return sx_set_error(fn_error(fn, "null logits"));
    if (!values_d) return sx_set_error(fn_error(fn, "null values"));
    if (max_nodes < 1) return sx_set_error(fn_error(fn, "max_nodes must be >= 1, got " + std::to_string(max_nodes)));
    const int logit_bytes = logits_dtype == SX_DTYPE_F32 ? 4 : logits_dtype == SX_DTYPE_BF16 || logits_dtype == SX_DTYPE_F16 ? 2 : 0;
    if (!logit_bytes) return sx_set_error(fn_error(fn, "unknown logits dtype " + std::to_string(logits_dtype)));
    if (L < 1 || L > SX_GUIDED_MAX_LEAVES)
        return sx_set_error(fn_error(fn, "leaves_per_tree must be in [1, 1024], got " + std::to_string(L)));
    if (num_envs <= 0) return 0;
    const DevConfig &d = cfg->dev;
    const int warp_bytes = carve_warp(d, nullptr, nullptr);
    const size_t smem = size_t(GUIDED_WARPS) * warp_bytes;
    const guided_backup_fn k = pick<guided_backup_fn>(cfg, sx_guided_backup_kernel<2, false>,
                                                      sx_guided_backup_kernel<4, false>, sx_guided_backup_kernel<4, true>,
                                                      sx_guided_backup_kernel<8, false>);
    const unsigned grid = unsigned((num_envs + GUIDED_WARPS - 1) / GUIDED_WARPS);
    k<<<grid, GUIDED_WARPS * 32, smem, static_cast<cudaStream_t>(stream)>>>(
        d, leaf_states.board, leaf_states.aux, leaf_states.captured, num_envs, max_nodes, L, tree, leaf_node_d,
        leaf_kind_d, static_cast<const uint8_t *>(logits_d), logits_dtype, logit_bytes, values_d, warp_bytes);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : fail("sx_guided_backup_kernel", e);
}

}  // namespace sx

extern "C" int sx_guided_select(const sx_config *cfg, sx_state st, int64_t num_envs, sx_guided_tree tree,
                                int32_t max_nodes, float c_puct, float fpu, sx_state leaf_states, int32_t *leaf_node_d,
                                int8_t *leaf_kind_d, void *stream)
{
    return sx::guided_select("sx_guided_select", cfg, st, num_envs, tree, max_nodes, c_puct, fpu, 1, 0.0f, nullptr,
                             leaf_states, leaf_node_d, leaf_kind_d, stream);
}

extern "C" int sx_guided_select_many(const sx_config *cfg, sx_state st, int64_t num_envs, sx_guided_tree tree,
                                     int32_t max_nodes, float c_puct, float fpu, int32_t leaves_per_tree,
                                     float virtual_loss, int32_t *inflight_d, sx_state leaf_states,
                                     int32_t *leaf_node_d, int8_t *leaf_kind_d, void *stream)
{
    return sx::guided_select("sx_guided_select_many", cfg, st, num_envs, tree, max_nodes, c_puct, fpu, leaves_per_tree,
                             virtual_loss, inflight_d, leaf_states, leaf_node_d, leaf_kind_d, stream);
}

extern "C" int sx_guided_backup(const sx_config *cfg, sx_state leaf_states, int64_t num_envs, sx_guided_tree tree,
                                int32_t max_nodes, const int32_t *leaf_node_d, const int8_t *leaf_kind_d,
                                const void *logits_d, int32_t logits_dtype, const float *values_d, void *stream)
{
    return sx::guided_backup("sx_guided_backup", cfg, leaf_states, num_envs, tree, max_nodes, 1, leaf_node_d,
                             leaf_kind_d, logits_d, logits_dtype, values_d, stream);
}

extern "C" int sx_guided_backup_many(const sx_config *cfg, sx_state leaf_states, int64_t num_envs,
                                     sx_guided_tree tree, int32_t max_nodes, int32_t leaves_per_tree,
                                     const int32_t *leaf_node_d, const int8_t *leaf_kind_d, const void *logits_d,
                                     int32_t logits_dtype, const float *values_d, void *stream)
{
    return sx::guided_backup("sx_guided_backup_many", cfg, leaf_states, num_envs, tree, max_nodes, leaves_per_tree,
                             leaf_node_d, leaf_kind_d, logits_d, logits_dtype, values_d, stream);
}
