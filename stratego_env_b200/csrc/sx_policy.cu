// sx_policy.cu -- masked-logit action sampling (the step right upstream of the env step in every rollout:
// examples/basic_game_loop.py:6-32 and README.md:38-65 of the reference build softmax(logits + log(mask + 1e-8))
// on the CPU and draw with np.random.choice, which costs 4x the env step there).
//
// One warp per game.  Exact categorical sampling by the Gumbel-max trick restricted to the valid entries:
//   action = argmax_{i : mask[i] != 0} (logits[i] / T - log(-log(u_i))),   u_i ~ U(0,1) from Philox4x32-10
// keyed by (seed, global env id, step, i), so results do not depend on placement.  Invalid entries have
// probability exactly 0 (the reference leaves them 1e-8 of relative mass).  Only the mask (1 byte / entry) is
// streamed; logits are fetched for valid entries only, so the kernel moves ~4 KB per game instead of ~19 KB.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"

namespace sx {

template <typename T>
__device__ __forceinline__ float load_logit(const T *p);
template <>
__device__ __forceinline__ float load_logit<float>(const float *p) { return *p; }
template <>
__device__ __forceinline__ float load_logit<__nv_bfloat16>(const __nv_bfloat16 *p) { return __bfloat162float(*p); }
template <>
__device__ __forceinline__ float load_logit<__half>(const __half *p) { return __half2float(*p); }

constexpr uint32_t RNG_POLICY = 0x504f4c59u;

// 23 random bits -> (k + 0.5) / 2^23: every value is exactly representable in float32 (k + 0.5 needs 24 significant
// bits) and lies strictly inside (0, 1), so -log(-log(u)) is always finite.  (24 bits + 0.5 rounds to 1.0 for the top
// value, which made that entry win regardless of its logit once in 2^24 draws.)
__host__ __device__ __forceinline__ float uniform_open01(uint32_t bits)
{
    return (float(bits >> 9) + 0.5f) * (1.0f / 8388608.0f);
}

// Gumbel-perturbed score z + G of one valid entry, G = -log(-log(u)) from the entry's Philox word.  The inner log needs
// relative accuracy: near u = 1, -log(u) is as small as 6e-8 while __logf promises only 3.6e-7 absolute there, and on
// the B200 it made G wrong by 1e-4 for u > 1 - 2^-10 and by 2.0 at the largest u, exactly the draws in which a low
// logit wins.  logf is accurate to a few ulp relative (G within 3e-6 for every u, tests/test_sampler_reference_gpu.py);
// the outer __logf's absolute error of 3.6e-7 is harmless.
__device__ __forceinline__ float gumbel_score(float z, uint32_t bits)
{
    return z - __logf(-logf(uniform_open01(bits)));
}

// One lane's share of a draw, the same in both samplers: the running argmax of the Gumbel-perturbed scores (a lane
// visits its entries in ascending index order, so `>` keeps the lowest index on ties) and, when LSE is set, the online
// log-sum-exp of z over the visited entries.  A z of -inf adds nothing to the sum and is skipped: in a lane that has
// not seen a finite z yet, exp(z - run_max) would be exp(-inf - -inf) = NaN and poison the whole warp's sum.
template <bool LSE>
struct GumbelMaxLane {
    float best = -INFINITY, best_logit = 0.0f;  // Gumbel-perturbed score of the running argmax and its scaled logit
    int best_i = -1;
    float run_max = -INFINITY, run_sum = 0.0f;

    __device__ __forceinline__ void visit(int i, float z, uint64_t gid, uint32_t step, uint2 key)
    {
        const uint4 r = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_POLICY ^ step, uint32_t(i)), key);
        const float score = gumbel_score(z, r.x);
        if (score > best || best_i < 0) { best = score; best_i = i; best_logit = z; }
        if (LSE) {
            if (z > run_max) { run_sum = run_sum * __expf(run_max - z) + 1.0f; run_max = z; }
            else if (z > -INFINITY) run_sum += __expf(z - run_max);
        }
    }

    // warp argmax (ties: lowest index, so the result is independent of the lane assignment) and log-sum-exp
    __device__ __forceinline__ void reduce_warp()
    {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float ob = __shfl_xor_sync(FULL, best, off), ol = __shfl_xor_sync(FULL, best_logit, off);
            const int oi = __shfl_xor_sync(FULL, best_i, off);
            const bool take = oi >= 0 && (best_i < 0 || ob > best || (ob == best && oi < best_i));
            if (take) { best = ob; best_i = oi; best_logit = ol; }
            if (LSE) {
                const float om = __shfl_xor_sync(FULL, run_max, off), os = __shfl_xor_sync(FULL, run_sum, off);
                const float nm = fmaxf(run_max, om);
                if (nm > -INFINITY) run_sum = run_sum * __expf(run_max - nm) + os * __expf(om - nm);
                run_max = nm;
            }
        }
    }

    // log p(best_i); NaN when every valid z is -inf (as torch.log_softmax)
    __device__ __forceinline__ float logprob() const { return best_logit - (run_max + __logf(run_sum)); }
};

template <typename T>
__global__ void __launch_bounds__(256) sx_sample_logits_kernel(const T *logits, const uint8_t *mask, long long num_envs,
                                                               int n_actions, long long env_base, uint2 key, uint32_t step,
                                                               float inv_temperature, int32_t *actions, float *logprob)
{
    const int lane = threadIdx.x & 31;
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= num_envs) return;
    const uint8_t *mrow = mask + env * n_actions;
    const T *lrow = logits + env * n_actions;
    const uint64_t gid = uint64_t(env_base + env);

    GumbelMaxLane<true> g;
    auto visit = [&](int i) { g.visit(i, load_logit<T>(lrow + i) * inv_temperature, gid, step, key); };

    // the mask row starts at env * n_actions: 4-byte aligned for every board (R*C*A is even x even or handled below)
    const int head = int((4 - (reinterpret_cast<uintptr_t>(mrow) & 3)) & 3);
    for (int i = lane; i < min(head, n_actions); i += 32)
        if (mrow[i]) visit(i);
    const int words = (n_actions - min(head, n_actions)) >> 2;
    const uint32_t *mw = reinterpret_cast<const uint32_t *>(mrow + head);
    // the mask words are fetched in batches of 8 independent loads per lane (8 x 32 words = 1 KB per batch) so that
    // the memory latency is paid once per batch instead of once per word; only valid entries cost a logit fetch
    constexpr int BATCH = 8;
    for (int w0 = 0; w0 < words; w0 += 32 * BATCH) {
        uint32_t m[BATCH];
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            const int w = w0 + 32 * j + lane;
            m[j] = w < words ? __ldg(mw + w) : 0u;
        }
#pragma unroll
        for (int j = 0; j < BATCH; ++j) {
            if (m[j] == 0) continue;
            const int base = head + ((w0 + 32 * j + lane) << 2);
#pragma unroll 1
            for (int b = 0; b < 4; ++b)
                if ((m[j] >> (8 * b)) & 0xff) visit(base + b);
        }
    }
    for (int i = head + (words << 2) + lane; i < n_actions; i += 32)
        if (mrow[i]) visit(i);

    g.reduce_warp();
    if (lane == 0) {
        actions[env] = g.best_i;  // -1: the mask had no valid entry
        if (logprob) logprob[env] = g.best_i >= 0 ? g.logprob() : 0.0f;
    }
}

// ---- the same draw straight from the game STATE ---------------------------------------------------------------------
// sx_sample_logits streams the 1-byte mask (3 700 bytes per 10x10 game) to find the ~14-25 valid entries.  The mask is a
// pure function of the compact state (~0.3 KB per game), so this kernel regenerates the mover's move sets from the state
// with the engine's own move generator (gen_moves: occupancy bit-lines), spreads the valid entries evenly over the lanes
// and runs the identical Gumbel-max / log-sum-exp per entry.  Same Philox key per (game, step, entry)
// and the same tie rule as the mask kernel, so both return the SAME action for the same key.

template <typename T, int K, bool LOGPROB, bool CM = false>
__global__ void __launch_bounds__(256) sx_sample_policy_kernel(const __grid_constant__ DevConfig cfg, const uint8_t *board,
                                                               const int16_t *aux, long long num_envs, long long env_base,
                                                               const T *logits, uint2 key, uint32_t step, float inv_temperature,
                                                               int32_t *actions, float *logprob, int warp_bytes)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
    if (env >= num_envs) return;
    uint8_t *warp_base = smem + size_t(warp) * warp_bytes;
    WarpMem m;
    const int slice = carve_warp(cfg, warp_base, &m);
    uint16_t *before = reinterpret_cast<uint16_t *>(warp_base + slice);  // [N] running move count per cell

    const uint32_t *gb = reinterpret_cast<const uint32_t *>(board + env * cfg.board_stride);
    {   // board_stride <= 256 bytes (K cells per lane, 32 lanes): at most K / 4 words per lane, no loop
        const int words = cfg.board_stride >> 2;
#pragma unroll
        for (int j = 0; j < (K + 3) / 4; ++j)
            if (lane + 32 * j < words) reinterpret_cast<uint32_t *>(m.board)[lane + 32 * j] = gb[lane + 32 * j];
    }
    const uint4 aw = *reinterpret_cast<const uint4 *>(aux + env * 8);
    Aux a;
    {
        const uint32_t w[4] = {aw.x, aw.y, aw.z, aw.w};
        aux_unpack(w, a);
    }
    __syncwarp();
    const bool any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);  // the mover's frame, like the mask (maenv:452-454)
    if (!any) {  // finished game or stuck player: the mask holds the noop entry [0,0,A-1] only (impl:514-515)
        if (lane == 0) {
            actions[env] = cfg.A - 1;
            if (logprob) logprob[env] = 0.0f;
        }
        return;
    }
    // Balance the entries over the lanes (an entry costs a Philox block and two transcendentals; a scout would pile a
    // dozen of them on one lane): moves are numbered 0 .. total-1 in ascending flat-index order, move t goes to lane
    // t % 32.  A lane finds its move's cell by binary search in the per-cell running count (shared memory) and the
    // channel as the r-th set bit of that cell's move set.
    int mine = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p < cfg.N) mine += __popc(m.moves[p].x) + __popc(m.moves[p].y);
    }
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, off);
        if (lane >= off) incl += v;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    {
        int run = incl - mine;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int p = lane * K + k;
            if (p < cfg.N) {
                before[p] = uint16_t(run);  // moves in cells < p
                run += __popc(m.moves[p].x) + __popc(m.moves[p].y);
            }
        }
    }
    __syncwarp();

    const T *lrow = logits + env * (long long)(cfg.N * cfg.A);
    const uint64_t gid = uint64_t(env_base + env);
    GumbelMaxLane<LOGPROB> g;
    for (int t = lane; t < total; t += 32) {  // ascending flat index within a lane, so `>` keeps the lowest index on ties
        int lo = 0, hi = cfg.N;               // last cell p with before[p] <= t: the cell that holds move t
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (int(before[mid]) <= t) lo = mid; else hi = mid;
        }
        const uint2 bits = m.moves[lo];
        const int ch = nth_set_bit64(bits, t - int(before[lo]));
        const int i = lo * cfg.A + ch;
        g.visit(i, load_logit<T>(lrow + i) * inv_temperature, gid, step, key);
    }
    g.reduce_warp();
    if (lane == 0) {
        actions[env] = g.best_i;
        if (LOGPROB) logprob[env] = g.logprob();
    }
}

// z = logit * (1 / T): a subnormal T makes 1 / T infinite and every 0-valued logit NaN
static bool valid_temperature(float temperature) { return temperature > 0.0f && 1.0f / temperature < INFINITY; }

}  // namespace sx

extern "C" int sx_sample_logits(const void *logits_d, int32_t logits_dtype, const uint8_t *mask_d, int64_t num_envs,
                                int32_t n_actions, int64_t env_base, uint64_t seed, uint32_t step, float temperature,
                                int32_t *actions_d, float *logprob_d, void *stream)
{
    using namespace sx;
    if (!logits_d || !mask_d || !actions_d) return sx_set_error("sx_sample_logits: null argument");
    if (!valid_temperature(temperature))
        return sx_set_error("sx_sample_logits: temperature must be > 0 with a finite reciprocal");
    if (n_actions < 1) return sx_set_error("sx_sample_logits: n_actions must be >= 1");
    if (num_envs <= 0) return 0;
    const int wpb = 8;
    const unsigned grid = unsigned((num_envs + wpb - 1) / wpb);
    const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float inv_t = 1.0f / temperature;
    switch (logits_dtype) {
    case SX_DTYPE_F32:
        sx_sample_logits_kernel<float><<<grid, wpb * 32, 0, s>>>(static_cast<const float *>(logits_d), mask_d, num_envs, n_actions,
                                                                 env_base, key, step, inv_t, actions_d, logprob_d);
        break;
    case SX_DTYPE_BF16:
        sx_sample_logits_kernel<__nv_bfloat16><<<grid, wpb * 32, 0, s>>>(static_cast<const __nv_bfloat16 *>(logits_d), mask_d,
                                                                         num_envs, n_actions, env_base, key, step, inv_t,
                                                                         actions_d, logprob_d);
        break;
    case SX_DTYPE_F16:
        sx_sample_logits_kernel<__half><<<grid, wpb * 32, 0, s>>>(static_cast<const __half *>(logits_d), mask_d, num_envs,
                                                                  n_actions, env_base, key, step, inv_t, actions_d, logprob_d);
        break;
    default:
        return sx_set_error("sx_sample_logits: unknown logits dtype");
    }
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : sx_set_error(std::string("sx_sample_logits_kernel: ") + cudaGetErrorString(e));
}

template <typename T>
static cudaError_t launch_policy(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const T *logits, uint2 key,
                                 uint32_t step, float inv_t, int32_t *actions, float *logprob, cudaStream_t s)
{
    using namespace sx;
    const DevConfig &d = cfg->dev;
    const int wpb = 8;
    const int warp_bytes = carve_warp(d, nullptr, nullptr) + round16(d.N * 2);
    const unsigned grid = unsigned((num_envs + wpb - 1) / wpb);
    const size_t smem = size_t(wpb) * warp_bytes;
    auto launch = [&](auto kernel) {
        kernel<<<grid, wpb * 32, smem, s>>>(d, st.board, st.aux, num_envs, env_base, logits, key, step, inv_t, actions, logprob,
                                            warp_bytes);
    };
    const bool lp = logprob != nullptr;
    if (d.N <= 64) lp ? launch(sx_sample_policy_kernel<T, 2, true>) : launch(sx_sample_policy_kernel<T, 2, false>);
    else if (d.N <= 128 && cfg->compact_movers)
        lp ? launch(sx_sample_policy_kernel<T, 4, true, true>) : launch(sx_sample_policy_kernel<T, 4, false, true>);
    else if (d.N <= 128) lp ? launch(sx_sample_policy_kernel<T, 4, true>) : launch(sx_sample_policy_kernel<T, 4, false>);
    else lp ? launch(sx_sample_policy_kernel<T, 8, true>) : launch(sx_sample_policy_kernel<T, 8, false>);
    return cudaGetLastError();
}

extern "C" int sx_sample_policy(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const void *logits_d,
                                int32_t logits_dtype, uint64_t seed, uint32_t step, float temperature, int32_t *actions_d,
                                float *logprob_d, void *stream)
{
    if (!cfg || !st.board || !st.aux || !logits_d || !actions_d) return sx_set_error("sx_sample_policy: null argument");
    if (!sx::valid_temperature(temperature))
        return sx_set_error("sx_sample_policy:temperature must be > 0 with a finite reciprocal");
    if (num_envs <= 0) return 0;
    const uint2 key = make_uint2(uint32_t(seed), uint32_t(seed >> 32));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const float inv_t = 1.0f / temperature;
    cudaError_t e;
    switch (logits_dtype) {
    case SX_DTYPE_F32:
        e = launch_policy(cfg, st, num_envs, env_base, static_cast<const float *>(logits_d), key, step, inv_t, actions_d, logprob_d, s);
        break;
    case SX_DTYPE_BF16:
        e = launch_policy(cfg, st, num_envs, env_base, static_cast<const __nv_bfloat16 *>(logits_d), key, step, inv_t, actions_d,
                          logprob_d, s);
        break;
    case SX_DTYPE_F16:
        e = launch_policy(cfg, st, num_envs, env_base, static_cast<const __half *>(logits_d), key, step, inv_t, actions_d, logprob_d, s);
        break;
    default:
        return sx_set_error("sx_sample_policy: unknown logits dtype");
    }
    return e == cudaSuccess ? 0 : sx_set_error(std::string("sx_sample_policy_kernel: ") + cudaGetErrorString(e));
}
