// sx_host.h -- host-side objects shared by the translation units of the library (not part of the C ABI).
#pragma once

#include <map>
#include <mutex>
#include <string>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"

struct LaunchPlan {
    int warps_per_block, blocks_per_sm, smem_per_block, num_sms, grid, regs;
    int warp_bytes, tile_bytes;
};

struct sx_config {
    sx::DevConfig dev;
    sx_layout layout;
    int cells_per_lane;  // K
    int games_per_warp;  // G
    int obs_elem_bytes = 4;  // 4: float32 observations; 2: bfloat16 / float16 (the LUT words of `dev` hold 16-bit patterns)
    bool compact_movers;  // gen_moves<.., COMPACT>: dense 10x10 boards (sx_device.cuh)
    bool compact_forced = false;  // sx_config_set_tuning chose compact_movers: it then applies to every launch mode
    sx_state start_states{nullptr, nullptr, nullptr};  // sx_config_set_start_states: curriculum table (device)
    long long n_start_states = 0;
    int32_t *start_index = nullptr;  // [env id - start_index_base] entry each game was started from (optional)
    long long start_index_base = 0, start_index_len = 0;
    int tune_warps = 0;   // sx_config_set_tuning: resident warps per SM of the warp-level kernel (0 = built-in choice)
    int tune_issue = -1;  // sx_config_set_tuning: where a game's background copy is issued (-1 = built-in choice)
    // launch shapes already worked out, keyed by (device, ops, mode): the occupancy / attribute queries cost tens
    // of microseconds, which matters for the one-game API
    mutable std::mutex plan_mutex;
    mutable std::map<uint64_t, LaunchPlan> plans;
};

int sx_set_error(const std::string &msg);  // records the text sx_last_error() returns; always returns -1
// true when p lies inside a live compressible allocation of sx_device_alloc (sx_alloc.cu)
bool sx_in_compressible_allocation(const void *p);

namespace sx {

// the instantiation of a one-warp-per-game search kernel (sx_expand.cu, sx_playout.cu, sx_search.cu, sx_guided.cu), as launch_policy
// (sx_policy.cu) picks it: cells per lane by board size, compact movers where configured
template <class F>
inline F pick(const sx_config *cfg, F k2, F k4, F k4cm, F k8)
{
    const int n = cfg->dev.N;
    return n <= 64 ? k2 : n <= 128 ? (cfg->compact_movers ? k4cm : k4) : k8;
}

inline int fail(const char *who, cudaError_t e) { return sx_set_error(std::string(who) + ": " + cudaGetErrorString(e)); }

inline bool null_state(const sx_state &s) { return !s.board || !s.aux || !s.captured; }

// expand and playout write the six step scalars of sx_outputs and nothing else
inline bool scalars_only(const sx_outputs &o)
{
    return !o.partial_obs && !o.full_obs && !o.valid_mask && !o.next_action && !o.terminal_partial_obs &&
           !o.terminal_full_obs;
}
constexpr const char *NOT_SCALARS_ONLY = ": only reward, done, winner, ending_invalid, illegal and player are written; "
                                         "observation, mask, next_action and terminal outputs must be null";

// the blocks of `threads` threads and `smem` bytes of shared memory that the current device holds at once, at most
// `wanted`, at least 1
template <class F>
inline cudaError_t resident_grid(F kernel, int threads, size_t smem, long long wanted, unsigned &grid)
{
    int device = 0, sms = 0, per_sm = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem);
    const long long most = (long long)(per_sm > 1 ? per_sm : 1) * sms;
    grid = unsigned(wanted < 1 ? 1 : wanted < most ? wanted : most);
    return e;
}

// the launch of a kernel of `warps`-warp blocks that take their games with claim_next (sx_device.cuh): the resident
// blocks, at most one per `warps` games, each with a contiguous range of per_block games, and no block without one
template <class F>
inline cudaError_t claim_grid(F kernel, int warps, size_t smem, long long num_envs, unsigned &grid, long long &per_block)
{
    const cudaError_t e = resident_grid(kernel, warps * 32, smem, (num_envs + warps - 1) / warps, grid);
    if (e != cudaSuccess) return e;
    per_block = (num_envs + grid - 1) / grid;
    grid = unsigned((num_envs + per_block - 1) / per_block);
    return e;
}

}  // namespace sx
