// sx_kernels.cu -- sm_100a kernels and C ABI of the B200 Stratego engine (include/stratego_b200.h).
//
// One persistent warp (or lane group, for the toy boards) per game.  The fused kernel stages a game's compact
// state in shared memory, applies the action, generates the next player's moves with occupancy bit-lines, and
// renders the outputs as "constant background image + sparse entries": the block's read-only background images
// go to HBM through the TMA engine (cp.async.bulk shared->global, ~30 KB per game for three instructions), the
// 50-250 state-dependent entries follow as plain stores that merge in L2.  No tensor cores, no CPU fallback.
// DESIGN.md section 3 has the design, the measurements behind each choice and the dead ends.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/stratego_b200.h"
#include "sx_device.cuh"
#include "sx_host.h"
#include "sx_toy.cuh"

namespace sx {

enum : uint32_t {
    OP_STEP = 1,         // decode + apply args.actions
    OP_MASK = 2,         // spatial mask -> out.valid_mask
    OP_PO = 4,           // partial observation -> out.partial_obs
    OP_FO = 8,           // full observation -> out.full_obs
    OP_RESET = 16,       // re-set envs selected by reset_mask before anything else
    OP_WRITE_STATE = 32, // store the state back
    OP_MASK_1D = 64,     // 1D mask straight to global (facade)
    OP_NEED_MOVES = 128  // run move generation even without a mask output (stuck check / sampler)
};

struct KernelArgs {
    DevConfig cfg;
    uint8_t *board;
    int16_t *aux;
    uint16_t *cap;
    long long num_envs, env_base;
    const int32_t *actions;
    int action_format;
    const int8_t *player_override;
    uint32_t flags, ops;  // flags: SX_* of the header in the low 16 bits, result-preserving tuning bits above (sx_step_all)
    sx_outputs out;
    uint8_t *mask1d;
    const uint8_t *setups;
    int n_setups;
    const int32_t *setup_idx;
    const uint8_t *reset_mask;
    uint2 key;
    long long *stats;
    const uint8_t *start_board;  // curriculum table (sx_config_set_start_states), n_start == 0: setups
    const int16_t *start_aux;
    const uint16_t *start_cap;
    uint32_t n_start;
    int32_t *start_index;  // [global env id - start_index_base], may be null
    long long start_index_base, start_index_len;
    int warp_bytes;  // shared-memory slice of one game (state + move sets + scratch)
    int tile_bytes;  // the block's background images (0 = this launch renders nothing)
};

// the block's background images: [partial obs][full obs][mask zeros + 16 bytes of alignment slack]
// EB = bytes per observation element (4, or 2 for the 16-bit observations)
template <int EB = 4>
__host__ __device__ inline int carve_tile(const DevConfig &cfg, uint32_t ops, uint8_t *base, Tile *t)
{
    int off = 0;
    if (t) t->po = reinterpret_cast<float *>(base + off);
    // three extra cell rows: the image is periodic in the cell (67 or 79 floats = 12 mod 16 bytes), so starting the
    // copy k rows in gives a source congruent mod 16 to ANY 4-byte aligned destination (5x5 and 15x15 observations
    // are not multiples of 16 bytes, so their rows in the output tensor are 4-, 8- or 12-byte misaligned); seven for
    // 16-bit elements, whose rows start at any even address (align_cells16)
    constexpr int extra = EB == 4 ? 3 : 7;
    off += (ops & OP_PO) ? round16((cfg.N + extra) * cfg.po_ch * EB) : 0;
    if (t) t->fo = reinterpret_cast<float *>(base + off);
    off += (ops & OP_FO) ? round16((cfg.N + extra) * cfg.fo_ch * EB) : 0;
    if (t) t->mask = base + off;
    off += (ops & OP_MASK) ? round16(cfg.mask_bytes + 16) : 0;
    return off;
}

// ---- output rendering ---------------------------------------------------------------------------------
// A game's observation is a per-variant constant "empty board" image (zeros in the one-hot planes, -1.0
// in the captured planes, 0.5 in the recent-move planes) plus 50-250 state-dependent entries, and its mask
// is zeros plus ~15-25 ones.  Each block keeps ONE read-only copy of those images in shared memory.  Per
// game, lane 0 hands the images to the TMA engine (cp.async.bulk shared -> global: ~30 KB of output for
// three instructions) at the top of the iteration, the warp runs the rule logic while the copy drains,
// and the sparse entries are then stored straight to global memory, where they merge with the freshly
// written lines in L2.  No warp owns a 30 KB tile, so shared memory no longer limits residency.
// Arguments and result by value so that the caller's state stays in registers.
template <int K, class GT, bool CM>
__device__ __noinline__ bool gen_moves_cold(const DevConfig *cfg, uint8_t *warp_base, uint4 auxw, int me)
{
    WarpMem m;
    carve_warp(*cfg, warp_base, &m);
    const uint32_t w[4] = {auxw.x, auxw.y, auxw.z, auxw.w};
    Aux a;
    aux_unpack(w, a);
    return gen_moves<K, GT, CM>(*cfg, m, a, me, false);
}

// Both players' observations of the game staged in the warp slice (its final position) into the terminal side buffers
// [env][player index 0 / 1][R][C][channels], same "background by TMA + sparse entries" rendering as the regular outputs.
// Out of line: a game ends once in hundreds of steps.
template <int K, class GT, class T = float>
static __device__ __noinline__ void render_terminal(const KernelArgs *args, const T *bg_po, const T *bg_fo,
                                                    uint8_t *warp_base, uint4 auxw, long long env, bool original)
{
    const DevConfig &cfg = args->cfg;
    WarpMem m;
    carve_warp(cfg, warp_base, &m);
    const uint32_t w[4] = {auxw.x, auxw.y, auxw.z, auxw.w};
    Aux a;
    aux_unpack(w, a);
    const ObsMap pom = original ? po_map_original() : po_map(), fom = original ? fo_map_original() : fo_map();
    T *tpo = reinterpret_cast<T *>(args->out.terminal_partial_obs), *tfo = reinterpret_cast<T *>(args->out.terminal_full_obs);
#pragma unroll 1
    for (int side = 0; side < 2; ++side) {
        T *gpo = tpo ? tpo + (env * 2 + side) * cfg.po_floats : nullptr;
        T *gfo = tfo ? tfo + (env * 2 + side) * cfg.fo_floats : nullptr;
        if constexpr (sizeof(T) == 2) {
            if (gpo) emit_obs16<GT>(gpo, bg_po, pom.channels, cfg.po_floats);
            if (gfo) emit_obs16<GT>(gfo, bg_fo, fom.channels, cfg.fo_floats);
        } else {
            if (gpo) {
                const int k = align_rows(pom.channels, int((reinterpret_cast<uintptr_t>(gpo) >> 2) & 3));
                emit_tile<GT>(reinterpret_cast<uint8_t *>(gpo), reinterpret_cast<const uint8_t *>(bg_po + k * pom.channels), cfg.po_floats * 4);
            }
            if (gfo) {
                const int k = align_rows(fom.channels, int((reinterpret_cast<uintptr_t>(gfo) >> 2) & 3));
                emit_tile<GT>(reinterpret_cast<uint8_t *>(gfo), reinterpret_cast<const uint8_t *>(bg_fo + k * fom.channels), cfg.fo_floats * 4);
            }
        }
        if (GT::lane() == 0) bulk_commit();
        GT::sync();  // commit_group and wait_group are kept apart (SX_TUNE_COMMIT_GAP)
        if (GT::lane() == 0) bulk_wait_all();
        GT::sync();
        if (original) {
            if (gpo) patch_obs<K, GT, true, T>(cfg, m, a, gpo, pom, side);
            if (gfo) patch_obs<K, GT, true, T>(cfg, m, a, gfo, fom, side);
        } else {
            if (gpo) patch_obs<K, GT, false, T>(cfg, m, a, gpo, pom, side);
            if (gfo) patch_obs<K, GT, false, T>(cfg, m, a, gfo, fom, side);
        }
        GT::sync();
    }
}

// MODE fixes the op set at compile time so that each hot launch type carries only its own code (the
// whole fused body is ~290 KB of SASS when everything is runtime-selected, far beyond the I-cache):
enum { MODE_GENERIC = 0, MODE_STEP_PO_MASK = 1, MODE_STEP_PO_FO_MASK = 2, MODE_STEP_LEAN = 3, MODE_MASK = 4, MODE_OBSERVE_PO_MASK = 5 };
constexpr uint32_t OPS_STEP_BASE = OP_STEP | OP_WRITE_STATE | OP_NEED_MOVES;

__host__ __device__ constexpr uint32_t mode_ops(int mode)
{
    return mode == MODE_STEP_PO_MASK ? (OPS_STEP_BASE | OP_PO | OP_MASK)
         : mode == MODE_STEP_PO_FO_MASK ? (OPS_STEP_BASE | OP_PO | OP_FO | OP_MASK)
         : mode == MODE_STEP_LEAN ? OPS_STEP_BASE
         : mode == MODE_MASK ? uint32_t(OP_MASK)
         : mode == MODE_OBSERVE_PO_MASK ? (OP_MASK | OP_PO) : 0u;
}

// end-of-run statistics (SURVEY.md section 5): games, wins per side, invalid endings, rejected actions, actions
// processed, attacks, setup draws.  Per-thread 32-bit counters of the thread-per-game kernel, published once per launch
struct StepCounters {
    uint32_t games, p1, p2, invalid, illegal, steps, attacks, resets;
    __device__ __forceinline__ void count_step(StepStatus status, bool done, const Aux &a)
    {
        if (status == STEP_ILLEGAL) illegal += 1;
        steps += 1;  // actions processed, accepted or not
        if (done && status != STEP_UNCHANGED) {
            games += 1;
            p1 += a.winner == 1;
            p2 += a.winner == -1;
            invalid += a.invalid;
        }
    }
    __device__ __forceinline__ void warp_sum()  // one game per lane (toy kernel): add the lanes' counters up
    {
        for (int off = 16; off > 0; off >>= 1) {
            games += __shfl_xor_sync(FULL, games, off); p1 += __shfl_xor_sync(FULL, p1, off);
            p2 += __shfl_xor_sync(FULL, p2, off); invalid += __shfl_xor_sync(FULL, invalid, off);
            illegal += __shfl_xor_sync(FULL, illegal, off); steps += __shfl_xor_sync(FULL, steps, off);
            attacks += __shfl_xor_sync(FULL, attacks, off); resets += __shfl_xor_sync(FULL, resets, off);
        }
    }
    __device__ __forceinline__ void publish(long long *stats) const
    {
        const uint32_t v[8] = {games, p1, p2, invalid, illegal, steps, attacks, resets};
#pragma unroll
        for (int i = 0; i < 8; ++i)
            if (v[i]) atomicAdd(reinterpret_cast<unsigned long long *>(stats + i), (unsigned long long)v[i]);
    }
};
// rare events of a step, added to the statistics right away by one lane (sx_fused_kernel)
__device__ __forceinline__ void count_rare(long long *stats, StepStatus status, bool done, const Aux &a)
{
    unsigned long long *s = reinterpret_cast<unsigned long long *>(stats);
    if (status == STEP_ILLEGAL) atomicAdd(s + 4, 1ull);
    if (done && status != STEP_UNCHANGED) {
        atomicAdd(s + 0, 1ull);
        if (a.winner == 1) atomicAdd(s + 1, 1ull);
        if (a.winner == -1) atomicAdd(s + 2, 1ull);
        if (a.invalid) atomicAdd(s + 3, 1ull);
    }
}
// out.illegal: 0 ok, 1 action rejected (game untouched), 2 the game's capture list overflowed (add_capture_inl)
__device__ __forceinline__ uint8_t illegal_code(StepStatus status, const Aux &a)
{
    return status == STEP_ILLEGAL ? 1 : (a.overflow ? 2 : 0);
}
constexpr int MAX_REDRAWS = 8;  // re-draws of an unplayable setup (first player without a move) per reset

// Result-preserving tuning bits the host sets per variant (sx_step_all): bits 20-21 = where a game's background copy is
// issued, bit 24 = SX_TUNE_COMMIT_GAP.
// SX_TUNE_COMMIT_GAP: on the boards that issue the copy LATE, `cp.async.bulk.commit_group` is directly followed by
// `cp.async.bulk.wait_group 0` (SASS: UTMACMDFLUSH; DEPBAR.LE SB0, 0 back to back), and that pair is slow on B200: ANY
// instruction between the two -- a warp sync, `nanosleep 0`, or the never-taken branches of the experiments build it
// was found with -- makes the 15x15 board 37 % faster (55 -> 75 M env-steps/s), 5x5
// 12 %, 6x6 6 %, 8x8 2 % (profiles/r2q_experiment_branch_layout_sweep.txt, r2r_commit_wait_gap.txt).  The 10x10 board
// with both observations is the one late-issue variant that does not gain (-1 %), so the host leaves the bit clear there.
constexpr uint32_t SX_TUNE_COMMIT_GAP = 0x1000000u;
// K = board cells per lane, G = games per warp (Grp<G>): 10x10 -> K 4, G 1; 3x4 / 4x4 -> K 2, G 4.
// Threads per block the kernel is compiled for (= its register budget: 65 536 / threads).  Everything with one game
// per warp gets 512 threads = 128 registers: with the 1 024-thread bound of round 1 the 6x6 / 8x8 kernels were held to
// 64 registers and spilled ~230 bytes per thread -- measured (profiles/r2l_small_board_launch_bound_sweep.txt) 8x8:
// 222 M env-steps/s at 1 024 threads / 16 warps, 242 M at 768 / 16, 272 M at 512 / 12; 6x6: 307 M / 337 M / 372 M.
// Several games per warp (3x4 ... 5x5) likewise: 5x5 385 M at 1 024 threads / 32 warps, 456 M at 768 / 24, 492 M at
// 512 / 16 (profiles/r2m_small_board_sweep.txt).
constexpr int FUSED_THREADS = 512;
// where the table entry a game is started from is recorded (sx_config_set_start_states); null = not recorded
__device__ __forceinline__ int32_t *start_index_slot(const KernelArgs &args, long long env)
{
    const long long i = args.env_base + env - args.start_index_base;
    return (args.start_index != nullptr && i >= 0 && i < args.start_index_len) ? args.start_index + i : nullptr;
}

// CM: gen_moves hands movers to lanes (dense 10x10 boards).  T: observation element, float or uint16_t (bfloat16 /
// float16 bit patterns); the 16-bit instantiations exist only for the modes that render observations.
template <int K, int MODE, int G, bool CM = false, class T = float>
__global__ void __launch_bounds__(FUSED_THREADS, 1)
sx_fused_kernel(const __grid_constant__ KernelArgs args)
{
    using GT = Grp<G>;
    extern __shared__ __align__(16) uint8_t smem[];
    const DevConfig &cfg = args.cfg;
    // `lane` is the lane within this game's group and `warp` the game slot within the block
    const int lane = GT::lane(), warp = (threadIdx.x >> 5) * G + GT::index(), warps_per_block = (blockDim.x >> 5) * G;
    const uint32_t ops = MODE == MODE_GENERIC ? args.ops : mode_ops(MODE), flags = args.flags;
    const int8_t *player_override =
        (MODE == MODE_GENERIC || MODE == MODE_MASK || MODE == MODE_OBSERVE_PO_MASK) ? args.player_override : nullptr;
    uint8_t *warp_base = smem + args.tile_bytes + size_t(warp) * args.warp_bytes;
    WarpMem m;
    carve_warp(cfg, warp_base, &m);

    const bool do_step = ops & OP_STEP, do_mask = ops & OP_MASK, do_po = ops & OP_PO, do_fo = ops & OP_FO;
    const bool do_tile = do_mask || do_po || do_fo;
    const bool do_sample = (flags & SX_SAMPLE_NEXT) && args.out.next_action != nullptr;
    const bool allow_osc = flags & SX_ALLOW_OSCILLATION;
    const bool need_moves = do_mask || do_sample || (ops & (OP_MASK_1D | OP_NEED_MOVES));
    const int mask_tile_bytes = round16(cfg.mask_bytes + 16);
    // the 32 / 33-channel 'original' observations run through the generic kernel only; the specialised hot modes keep
    // compile-time channel maps
    const bool original = MODE == MODE_GENERIC && cfg.original_channels != 0;
    const ObsMap pom = original ? po_map_original() : po_map(), fom = original ? fo_map_original() : fo_map();

    // the block's read-only background images
    Tile bg;
    carve_tile<sizeof(T)>(cfg, ops, smem, &bg);
    if (do_tile) {
        // + 3 (7) rows: see carve_tile
        if (do_po) fill_background<T>(cfg, reinterpret_cast<T *>(bg.po), pom, threadIdx.x, blockDim.x, cfg.N + bg_extra_cells<T>());
        if (do_fo) fill_background<T>(cfg, reinterpret_cast<T *>(bg.fo), fom, threadIdx.x, blockDim.x, cfg.N + bg_extra_cells<T>());
        if (do_mask)
            for (int i = threadIdx.x; i < (mask_tile_bytes >> 4); i += blockDim.x)
                reinterpret_cast<uint4 *>(bg.mask)[i] = make_uint4(0, 0, 0, 0);
        fence_async_smem();  // generic-proxy writes above -> visible to the TMA engine (async proxy)
    }
    __syncthreads();

    // ---- software pipeline -----------------------------------------------------------------------------
    // While game i runs, (1) game i+1's state / action loads are in flight in registers and (2) game i+1's
    // background images are already on their way to HBM: they are issued BEFORE waiting for game i's copy,
    // so a warp keeps up to two bulk groups in flight and never idles on TMA completion.
    struct Prefetched {
        uint32_t board[2], cap[4];
        uint4 aux;
        int action;
    };
    const int board_words = cfg.board_stride >> 2, cap_words = cfg.cap_stride >> 1;
    auto load_state = [&](long long e, Prefetched &pf) {
        const uint32_t *gb = reinterpret_cast<const uint32_t *>(args.board + e * cfg.board_stride);
        const uint32_t *gc = reinterpret_cast<const uint32_t *>(args.cap + e * cfg.cap_stride);
#pragma unroll
        for (int j = 0; j < 2; ++j) pf.board[j] = lane + GT::L * j < board_words ? gb[lane + GT::L * j] : 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) pf.cap[j] = lane + GT::L * j < cap_words ? gc[lane + GT::L * j] : 0u;
        pf.aux = *reinterpret_cast<const uint4 *>(args.aux + e * 8);
        pf.action = do_step ? args.actions[e] : 0;
    };
    auto issue_background = [&](long long e) {
        // the small mask copy goes first (measured: +3 % over observation-first at 10 warps per SM)
        if (do_mask) {
            uint8_t *gmask = args.out.valid_mask + e * cfg.mask_bytes;
            emit_tile<GT>(gmask, bg.mask + (reinterpret_cast<uintptr_t>(gmask) & 15), cfg.mask_bytes);
        }
        if constexpr (sizeof(T) == 2) {
            if (do_po) emit_obs16<GT>(reinterpret_cast<T *>(args.out.partial_obs) + e * cfg.po_floats, reinterpret_cast<const T *>(bg.po), pom.channels, cfg.po_floats);
            if (do_fo) emit_obs16<GT>(reinterpret_cast<T *>(args.out.full_obs) + e * cfg.fo_floats, reinterpret_cast<const T *>(bg.fo), fom.channels, cfg.fo_floats);
        } else {
            if (do_po) {
                float *g = args.out.partial_obs + e * cfg.po_floats;
                const int k = align_rows(pom.channels, int((reinterpret_cast<uintptr_t>(g) >> 2) & 3));
                emit_tile<GT>(reinterpret_cast<uint8_t *>(g), reinterpret_cast<const uint8_t *>(bg.po + k * pom.channels),
                              cfg.po_floats * 4);
            }
            if (do_fo) {
                float *g = args.out.full_obs + e * cfg.fo_floats;
                const int k = align_rows(fom.channels, int((reinterpret_cast<uintptr_t>(g) >> 2) & 3));
                emit_tile<GT>(reinterpret_cast<uint8_t *>(g), reinterpret_cast<const uint8_t *>(bg.fo + k * fom.channels),
                              cfg.fo_floats * 4);
            }
        }
        if (lane == 0) bulk_commit();
    };

    // statistics: a finished game, a rejected action or a (re)draw are rare and go straight to the counters (one lane,
    // one atomic each); attacks and the step count stay in registers / are derived, and are published once per launch.
    // (Eight live counters cost the 64-register kernels of the small boards 30 % more spill traffic.)
    uint32_t n_attacks = 0, n_steps = 0;
    // Game g goes to game slot g mod (slots in the grid).  (Runs of 8 or 32 consecutive games per slot measured -1 to
    // -3 %, profiles/r2u_chunk_mapping_sweep.txt.)
    const int total_warps = gridDim.x * warps_per_block;  // (a 64-bit stride made the ptxas allocation spill more)
    long long env = (long long)blockIdx.x * warps_per_block + warp;
    Prefetched pf;
    // Where a game's background copy is issued.  The sparse entries must reach L2 while the background lines are
    // still resident there (otherwise every 4-byte store becomes a DRAM read-modify-write; measured: storing them one
    // whole game later costs 10-25 %), and the warp should have work to do while its copy drains.  0 = late, right
    // before the wait; 1 = after the outcome, before state write-back and sampling (best for a 10x10 board with one
    // observation: ~400 instructions overlap the drain); 2 = top of the game.  sx_step_all picks per variant
    // (sx_config_set_tuning overrides).
    const int issue_at = (flags >> 20) & 3;
    if (env < args.num_envs) load_state(env, pf);
    for (; env < args.num_envs; env += total_warps) {
        const uint64_t gid = uint64_t(args.env_base + env);
        // ---- this game's state has arrived in registers: move it to the working slice, request the next ----
        GT::sync();
#pragma unroll
        for (int j = 0; j < 2; ++j)
            if (lane + GT::L * j < board_words) reinterpret_cast<uint32_t *>(m.board)[lane + GT::L * j] = pf.board[j];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (lane + GT::L * j < cap_words) reinterpret_cast<uint32_t *>(m.cap)[lane + GT::L * j] = pf.cap[j];
        const int action = pf.action;
        Aux a;
        {
            const uint32_t w[4] = {pf.aux.x, pf.aux.y, pf.aux.z, pf.aux.w};
            aux_unpack(w, a);
        }
        GT::sync();
        const long long next_env = env + total_warps;
        const bool has_next = next_env < args.num_envs;
        if (has_next) load_state(next_env, pf);
        if (do_tile && issue_at == 2) issue_background(env);

        bool dirty = false;
        // out-of-line helpers take and return everything by value so that `a` never has to live in local memory
        // (Re)starts the game: episode number `episode` (games this env has started so far), draw number `attempt`.
        // maenv:530-534: every second game repeats the previous setup seen from the other side; maenv:352-354: one setup
        // for every game of this env.  Both are choices of WHICH Philox counter the draw uses (ResetSource).
        auto do_reset = [&](uint32_t episode, int attempt) {
            GT::sync();
            const bool other_side = (flags & SX_REPEAT_OTHER_SIDE) && (episode & 1u);
            const uint32_t rng_episode = (flags & SX_SAME_SETUP) ? 0u : other_side ? episode - 1u : episode;
            const uint32_t draw = uint32_t(attempt) | (other_side ? 256u : 0u) | ((flags & SX_RESET_RANDOM_SHUFFLE) ? 512u : 0u);
            const uint4 nw = args.n_start != 0
                ? reset_from_table<GT>(&cfg, warp_base, args.start_board, args.start_aux, args.start_cap, args.n_start,
                                       uint32_t(attempt), args.key, gid, episode, (flags & SX_SAME_SETUP) ? 0u : episode,
                                       start_index_slot(args, env))
                : reset_game<GT>(&cfg, warp_base, args.setups, args.n_setups,
                                 args.setup_idx ? args.setup_idx + env * 2 : nullptr, draw, args.key, gid, episode, rng_episode);
            const uint32_t w[4] = {nw.x, nw.y, nw.z, nw.w};
            aux_unpack(w, a);
        };
        auto regen_moves = [&](int me) -> bool {
            uint32_t w[4];
            aux_pack(a, w);
            GT::sync();
            return gen_moves_cold<K, GT, CM>(&cfg, warp_base, make_uint4(w[0], w[1], w[2], w[3]), me);
        };
        if (MODE == MODE_GENERIC && (ops & OP_RESET) && (args.reset_mask == nullptr || args.reset_mask[env] != 0)) {
            // drawn setups only (explicit setup_idx rows are the caller's choice): see the auto-reset below
            const uint32_t episode = a.episode;
#pragma unroll 1
            for (int tries = 0; tries < MAX_REDRAWS; ++tries) {
                do_reset(episode, tries);
                if (args.setup_idx != nullptr || regen_moves(a.to_move)) break;
            }
            dirty = true;
        }

        // ---- step: decode, validate, apply (impl:897-1028) ----------------------------------------
        StepStatus status = STEP_UNCHANGED;
        const int mover = a.to_move;
        if (do_step) {
            Move mv = args.action_format == SX_ACTION_SPATIAL ? decode_spatial(cfg, action, mover) : decode_1d(cfg, action);
            if (mv.noop && !mv.bad && !a.over) {  // impl:809-814
                if (regen_moves(mover)) mv.bad = true;
            }
            int attack;
            status = apply_move<GT>(cfg, m, a, mv, allow_osc, attack);
            dirty |= status != STEP_ILLEGAL;
            n_attacks += attack;
            n_steps += 1;
        }

        // ---- move list of the player the outputs are for -------------------------------------------
        int viewer = a.to_move;
        if (player_override) viewer = player_override[env] == 1 ? 0 : 1;
        bool any = false;
        const bool have_moves = need_moves && (status == STEP_MOVED || !do_step || do_mask || do_sample || (ops & OP_MASK_1D));
        if (have_moves) any = gen_moves<K, GT, CM>(cfg, m, a, viewer, false);

        if (status == STEP_MOVED) {
            if (have_moves && !any && !a.over) { a.over = 1; a.winner = mover == 0 ? 1 : -1; }  // impl:1031-1036
            if (a.turn >= a.max_turns && !a.over) {  // impl:1040-1043
                a.over = 1;
                a.invalid = 1;
                if (have_moves && any) any = regen_moves(viewer);  // terminal: noop only
            }
        }
        const bool done = do_step && status != STEP_ILLEGAL && a.over;
        if (do_step) {
            if (lane == 0) {
                const int w = a.winner;
                if (args.out.done) args.out.done[env] = done ? 1 : 0;
                if (args.out.winner) args.out.winner[env] = int8_t(done ? w : 0);
                if (args.out.ending_invalid) args.out.ending_invalid[env] = (done && a.invalid) ? 1 : 0;
                if (args.out.illegal) args.out.illegal[env] = illegal_code(status, a);
                if (args.out.reward) args.out.reward[env] = (done && !a.invalid) ? float(w) : 0.0f;  // maenv:777-801
            }
            if (args.stats && lane == 0 && (status == STEP_ILLEGAL || done)) count_rare(args.stats, status, done, a);
        }

        // maenv:772-773 hands BOTH players their observation of the finished game; with auto-reset the regular outputs
        // already show the next game, so the terminal observations go to side buffers (cold path).
        if (done && (args.out.terminal_partial_obs != nullptr || args.out.terminal_full_obs != nullptr)) {
            uint32_t w[4];
            aux_pack(a, w);
            GT::sync();
            render_terminal<K, GT, T>(&args, reinterpret_cast<const T *>(bg.po), reinterpret_cast<const T *>(bg.fo), warp_base, make_uint4(w[0], w[1], w[2], w[3]), env, original);
        }
        if (done && (flags & SX_AUTO_RESET)) {
            // A drawn setup in which the player to move has no move cannot be played in the reference either (the only
            // entry of its mask is the noop, which maenv.step rejects: impl:316-347 decodes it to an illegal move), so
            // such a draw -- 2e-6 of Standard shuffles, none of the human tables -- is drawn again (next attempt number).
            const uint32_t episode = a.episode;
#pragma unroll 1  // (unrolled eight times this loop alone made the hot kernels 20 % bigger and the small boards 15-25 % slower)
            for (int tries = 0; tries < MAX_REDRAWS; ++tries) {
                do_reset(episode, tries);
                if (args.stats && lane == 0) atomicAdd(reinterpret_cast<unsigned long long *>(args.stats + 7), 1ull);
                viewer = a.to_move;
                if (!need_moves) break;
                any = regen_moves(viewer);
                if (any) break;
            }
        }
        if (args.out.player && lane == 0) args.out.player[env] = viewer == 0 ? 1 : -1;
        if (do_tile && issue_at == 1) issue_background(env);

        if ((ops & OP_MASK_1D) != 0) {
            uint8_t *row = args.mask1d + env * cfg.action_size;
            mark_1d_global<K, GT>(&cfg, m.moves, viewer, row);
            if (!any && lane == 0) row[cfg.action_size - 1] = 1;  // impl:639-640
        }

        if ((ops & OP_WRITE_STATE) && dirty) {
            uint32_t *gb = reinterpret_cast<uint32_t *>(args.board + env * cfg.board_stride);
            for (int i = lane; i < (cfg.board_stride >> 2); i += GT::L) gb[i] = reinterpret_cast<const uint32_t *>(m.board)[i];
            uint32_t *gc = reinterpret_cast<uint32_t *>(args.cap + env * cfg.cap_stride);
            for (int i = lane; i < (cfg.cap_stride >> 1); i += GT::L) gc[i] = reinterpret_cast<const uint32_t *>(m.cap)[i];
            if (lane == 0) {
                uint32_t w[4];
                aux_pack(a, w);
                *reinterpret_cast<uint4 *>(args.aux + env * 8) = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }

        if (do_sample) {
            const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SAMPLE ^ uint32_t(a.turn), a.episode), args.key);
            const int act = sample_move<K, GT>(cfg, m, any, rnd.x);
            if (lane == 0) args.out.next_action[env] = act;
        }

        // ---- render: sparse entries on top of the (by now written) background ---------------------------
        if (do_tile && issue_at == 0) {
            issue_background(env);
            if (flags & SX_TUNE_COMMIT_GAP) GT::sync();  // keeps commit_group and wait_group apart (see SX_TUNE_COMMIT_GAP)
        }
        if (do_tile) {
            if (lane == 0) bulk_wait_all();  // this game's background is in global memory
            GT::sync();
            if (original) {
                if (do_po) patch_obs<K, GT, true, T>(cfg, m, a, reinterpret_cast<T *>(args.out.partial_obs) + env * cfg.po_floats, pom, viewer);
                if (do_fo) patch_obs<K, GT, true, T>(cfg, m, a, reinterpret_cast<T *>(args.out.full_obs) + env * cfg.fo_floats, fom, viewer);
            } else {
                if (do_po) patch_obs<K, GT, false, T>(cfg, m, a, reinterpret_cast<T *>(args.out.partial_obs) + env * cfg.po_floats, pom, viewer);
                if (do_fo) patch_obs<K, GT, false, T>(cfg, m, a, reinterpret_cast<T *>(args.out.full_obs) + env * cfg.fo_floats, fom, viewer);
            }
            if (do_mask) {
                uint8_t *gmask = args.out.valid_mask + env * cfg.mask_bytes;
                mark_spatial<K, GT>(cfg, m, gmask);
                if (!any && lane == 0) *(gmask + cfg.A - 1) = 1;  // [0,0,A-1], impl:514-515
            }
        }
        GT::sync();
    }

    if (args.stats && lane == 0) {  // all lanes of a game carry identical counters
        if (n_steps) atomicAdd(reinterpret_cast<unsigned long long *>(args.stats + 5), (unsigned long long)n_steps);
        if (n_attacks) atomicAdd(reinterpret_cast<unsigned long long *>(args.stats + 6), (unsigned long long)n_attacks);
    }
}


// ---- toy boards: one thread per game (sx_toy.cuh has the design) ------------------------------------------------------
// shared memory: [block background images][per warp: stage 32 x 48 B | mask image of 32 rows | two observation tiles]
// Measured (profiles/r1l_*): throughput follows the number of resident warps (8: 0.87 G, 12: 1.23 G, 16: 1.43 G
// env-steps/s on Micro), not the number of tiles per warp (2, 4, 8, 16 tiles: same), so the launch keeps two tiles and
// as many warps as shared memory holds.
// compiled for the 12 warps it runs with: 144 registers instead of the 120 a 512-thread bound leaves (Micro +1 %, Tiny
// +4 %, profiles/r2o_toy_register_budget_sweep.txt)
constexpr int TOY_TILES = 2;  // observation tiles per warp: one is rendered while the copy of the other is read; divides 32
constexpr int TOY_THREADS = 384;
// T: observation element, float or uint16_t (bfloat16 / float16 bit patterns)
template <int MODE, class T = float>
__global__ void __launch_bounds__(TOY_THREADS, 1) sx_toy_kernel(const __grid_constant__ KernelArgs args)
{
    using GT = Grp<1>;
    extern __shared__ __align__(16) uint8_t smem[];
    const DevConfig &cfg = args.cfg;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    constexpr uint32_t ops = mode_ops(MODE);
    constexpr bool do_mask = (ops & OP_MASK) != 0, do_po = (ops & OP_PO) != 0, do_fo = (ops & OP_FO) != 0;
    constexpr bool do_tile = do_mask || do_po || do_fo;
    constexpr bool half = sizeof(T) == 2;
    const uint32_t flags = args.flags;
    const bool do_sample = (flags & SX_SAMPLE_NEXT) && args.out.next_action != nullptr;
    const bool allow_osc = flags & SX_ALLOW_OSCILLATION;
    const ObsMap pom = po_map(), fom = fo_map();

    Tile bg;
    carve_tile<sizeof(T)>(cfg, ops, smem, &bg);
    if (do_tile) {
        if (do_po) fill_background<T>(cfg, reinterpret_cast<T *>(bg.po), pom, threadIdx.x, blockDim.x, cfg.N + bg_extra_cells<T>());
        if (do_fo) fill_background<T>(cfg, reinterpret_cast<T *>(bg.fo), fom, threadIdx.x, blockDim.x, cfg.N + bg_extra_cells<T>());
    }
    __syncthreads();

    uint8_t *const stage = smem + args.tile_bytes + size_t(warp) * args.warp_bytes;
    uint8_t *const mask_img = stage + toy::GAMES * toy::STAGE_BYTES;
    const int mask_total = toy::GAMES * cfg.mask_bytes;
    const int mask_img_bytes = do_mask ? round16(mask_total + 16) : 0;
    uint8_t *const tiles = mask_img + mask_img_bytes;
    const int po_bytes = do_po ? cfg.po_floats * int(sizeof(T)) : 0, fo_bytes = do_fo ? cfg.fo_floats * int(sizeof(T)) : 0;
    // 16-bit rows are 8 mod 16 bytes long on the 12-cell board (toy::tile_slot), so a tile starts at the residue its
    // games' rows have in the output tensor; float32 rows of these boards are whole multiples of 16 bytes
    const int po_slot = half ? toy::tile_slot(po_bytes) : po_bytes, fo_slot = half ? toy::tile_slot(fo_bytes) : fo_bytes;
    const int tile_stride = po_slot + fo_slot;
    // the warp's two observation tiles hold the background image for the whole launch
    // T tiles per warp.  Measured and not kept (profiles/r1l_toy_sweeps.txt, r2g_*, r2x_*, r2y_*): 4 or 8 tiles per warp
    // (Micro 1 198 M / 847 M vs 1 448 M env-steps/s), two or four consecutive games per tile set leaving as ONE larger bulk
    // copy (1 234 M / 914 M), two games rendered per pass by the half-warps (1 360 M).  Every one of them needs more
    // shared memory per warp, and the block's shared memory comes out of the SM's 256 KB L1: this kernel keeps ~100 bytes
    // of per-thread arrays in local memory, so it wants the L1 that 150 KB of shared memory leaves.
    constexpr int NT = TOY_TILES;
    uint32_t undo_po[NT], undo_fo[NT];
#pragma unroll
    for (int h = 0; h < NT; ++h) undo_po[h] = undo_fo[h] = lane < 16 ? 0u : toy::UNDO_NONE;  // cell lanes: "channel 0" four times
    for (int h = 0; h < NT; ++h) {
        if constexpr (half) {  // tiles 8-byte aligned (tile_slot), rows a multiple of 8 bytes (cells a multiple of 4)
            if (do_po)
                for (int i = lane; i < (po_bytes >> 3); i += 32)
                    reinterpret_cast<uint2 *>(tiles + h * tile_stride + ((h * po_bytes) & 15))[i] = reinterpret_cast<const uint2 *>(bg.po)[i];
            if (do_fo)
                for (int i = lane; i < (fo_bytes >> 3); i += 32)
                    reinterpret_cast<uint2 *>(tiles + h * tile_stride + po_slot + ((h * fo_bytes) & 15))[i] = reinterpret_cast<const uint2 *>(bg.fo)[i];
        } else {
            if (do_po)
                for (int i = lane; i < (po_bytes >> 4); i += 32)
                    reinterpret_cast<uint4 *>(tiles + h * tile_stride)[i] = reinterpret_cast<const uint4 *>(bg.po)[i];
            if (do_fo)
                for (int i = lane; i < (fo_bytes >> 4); i += 32)
                    reinterpret_cast<uint4 *>(tiles + h * tile_stride + po_bytes)[i] = reinterpret_cast<const uint4 *>(bg.fo)[i];
        }
    }
    __syncwarp();

    const toy::Geometry geo = toy::make_geometry(cfg);
    StepCounters cnt{};
    const long long n_groups = args.num_envs / toy::GAMES;
    // the next group's state loads are issued before this group is rendered, so they never stall the rules
    uint4 pf_b = make_uint4(0, 0, 0, 0), pf_c = pf_b, pf_a = pf_b;
    int pf_action = 0;
    auto load_state = [&](long long e) {
        pf_b = *reinterpret_cast<const uint4 *>(args.board + e * 16);
        pf_c = *reinterpret_cast<const uint4 *>(args.cap + e * 8);
        pf_a = *reinterpret_cast<const uint4 *>(args.aux + e * 8);
        pf_action = args.actions[e];
    };
    const long long group_stride = (long long)gridDim.x * wpb;
    if ((long long)blockIdx.x * wpb + warp < n_groups) load_state(((long long)blockIdx.x * wpb + warp) * toy::GAMES + lane);
    for (long long group = (long long)blockIdx.x * wpb + warp; group < n_groups; group += group_stride) {
        const long long env0 = group * toy::GAMES, env = env0 + lane;
        const uint64_t gid = uint64_t(args.env_base + env);
        if (do_tile) {
            // the mask image is about to be rewritten: its copy is the OLDEST group of the previous 32 games, so it is
            // enough that all but the newest T - 1 groups (the last observation tiles, which the render loop below waits
            // for tile by tile) have been read; draining everything here stalled the warp once per 32 games (Micro +1 %)
            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(TOY_TILES - 1) : "memory");
            __syncwarp();
            if (do_mask)
                for (int i = lane; i < (mask_img_bytes >> 4); i += 32) reinterpret_cast<uint4 *>(mask_img)[i] = make_uint4(0, 0, 0, 0);
        }
        // ---- this thread's game: 48 bytes of state in registers (requested one group ahead) --------------------------
        toy::State s;
        s.b[0] = pf_b.x; s.b[1] = pf_b.y; s.b[2] = pf_b.z; s.b[3] = pf_b.w;
        s.c[0] = pf_c.x; s.c[1] = pf_c.y; s.c[2] = pf_c.z; s.c[3] = pf_c.w;
        Aux a;
        {
            const uint32_t w[4] = {pf_a.x, pf_a.y, pf_a.z, pf_a.w};
            aux_unpack(w, a);
        }
        const int action = pf_action;
        toy::MoveSets mv;

        // ---- step: decode, validate, apply (impl:897-1028) ----------------------------------------------------
        const int mover = a.to_move;
        Move move = args.action_format == SX_ACTION_SPATIAL ? decode_spatial(cfg, action, mover) : decode_1d(cfg, action);
        StepStatus status = STEP_ILLEGAL;
        bool done = false;
        int viewer = 0, total = 0;
        uint32_t reset_episode = 0;
        // Move generation is ONE inlined copy run up to three times: pass 0 only for a noop action (legal only when
        // nothing else is, impl:809-814), pass 1 for the next player (stuck check, impl:1031-1036), pass 2 for the fresh
        // game of an auto-reset.
#pragma unroll 1
        for (int pass = (move.noop && !move.bad && !a.over) ? 0 : 1; pass < 2 + MAX_REDRAWS; ++pass) {
            if (pass == 1) {
                const uint32_t end_before = move.bad || move.noop ? 0u : toy::cell_get(s, move.end);
                status = toy::apply_move(cfg, s, a, move, allow_osc);
                cnt.attacks += (status == STEP_MOVED && (end_before & CELL_RANK) != 0) ? 1 : 0;
                viewer = a.to_move;
            }
            if (pass >= 2) {  // (re)draw the fresh game: attempt pass - 2 of episode reset_episode (ONE inlined copy of the reset)
                a.episode = reset_episode;
                toy::reset_game(cfg, s, a, args.setups, args.n_setups, (flags & SX_RESET_RANDOM_SHUFFLE) != 0, args.key, gid,
                                (flags & SX_SAME_SETUP) ? 0u : reset_episode, uint32_t(pass - 2));
                cnt.resets += 1;
                viewer = a.to_move;
            }
            const int who = pass == 0 ? mover : viewer;
            total = toy::gen_moves(cfg, geo, s, a, who, false, mv);
            if (pass == 0) {
                if (total > 0) move.bad = true;
                continue;
            }
            if (pass >= 2) {  // an unplayable draw (first player without a move) is drawn again, see sx_fused_kernel
                if (total > 0 || pass - 1 >= MAX_REDRAWS) break;
                continue;
            }
            if (status == STEP_MOVED) {
                if (total == 0 && !a.over) { a.over = 1; a.winner = mover == 0 ? 1 : -1; }
                if (a.turn >= a.max_turns && !a.over) {  // impl:1040-1043; terminal masks are noop-only
                    a.over = 1;
                    a.invalid = 1;
                    total = 0;
                    toy::clear_sets(mv);
                }
            }
            done = status != STEP_ILLEGAL && a.over;
            const int w = a.winner;
            if (args.out.done) args.out.done[env] = done ? 1 : 0;
            if (args.out.winner) args.out.winner[env] = int8_t(done ? w : 0);
            if (args.out.ending_invalid) args.out.ending_invalid[env] = (done && a.invalid) ? 1 : 0;
            if (args.out.illegal) args.out.illegal[env] = illegal_code(status, a);
            if (args.out.reward) args.out.reward[env] = (done && !a.invalid) ? float(w) : 0.0f;  // maenv:777-801
            cnt.count_step(status, done, a);
            if (!(done && (flags & SX_AUTO_RESET))) break;
            reset_episode = a.episode;  // the next pass draws the new game
        }
        if (args.out.player) args.out.player[env] = viewer == 0 ? 1 : -1;

        // ---- state write-back, uniform valid-action sample -----------------------------------------------------
        *reinterpret_cast<uint4 *>(args.board + env * 16) = make_uint4(s.b[0], s.b[1], s.b[2], s.b[3]);
        *reinterpret_cast<uint4 *>(args.cap + env * 8) = make_uint4(s.c[0], s.c[1], s.c[2], s.c[3]);
        {
            uint32_t w[4];
            aux_pack(a, w);
            *reinterpret_cast<uint4 *>(args.aux + env * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        if (do_sample) {
            const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SAMPLE ^ uint32_t(a.turn), a.episode), args.key);
            args.out.next_action[env] = toy::pick_move(cfg, mv, total, rnd.x);
        }
        if (group + group_stride < n_groups) load_state((group + group_stride) * toy::GAMES + lane);
        if (!do_tile) continue;

        // ---- render the warp's 32 games ------------------------------------------------------------------------
        uint8_t *gmask = do_mask ? args.out.valid_mask + env0 * cfg.mask_bytes : nullptr;
        uint8_t *mask_rows = mask_img + (reinterpret_cast<uintptr_t>(gmask) & 15);  // source congruent to the destination mod 16
        __syncwarp();  // the mask image is zero
        if (do_mask) {
            uint8_t *row = mask_rows + lane * cfg.mask_bytes;
            toy::mark_row(cfg, mv, row);
            if (total == 0) row[cfg.A - 1] = 1;  // [0,0,A-1], impl:514-515
        }
        {
            uint8_t *st = stage + lane * toy::STAGE_BYTES;
            *reinterpret_cast<uint4 *>(st) = make_uint4(s.b[0], s.b[1], s.b[2], s.b[3]);
            *reinterpret_cast<uint4 *>(st + 16) = make_uint4(s.c[0], s.c[1], s.c[2], s.c[3]);
            *reinterpret_cast<uint32_t *>(st + 32) = uint32_t(a.rfrom[0]) | (uint32_t(a.rto[0]) << 8) | (uint32_t(a.rfrom[1]) << 16) |
                                                      (uint32_t(a.rto[1]) << 24);
            *reinterpret_cast<uint32_t *>(st + 36) = uint32_t(a.rcode[0]) | (uint32_t(a.rcode[1]) << 4) | (uint32_t(a.ncap) << 8) |
                                                      (uint32_t(viewer) << 16);
        }
        fence_async_smem();
        __syncwarp();
        if (do_mask) {  // the 32 mask rows are contiguous in the output tensor: one bulk copy (+ unaligned head / tail words)
            emit_tile<GT>(gmask, mask_rows, mask_total);
            if (lane == 0) bulk_commit();
        }
        if (do_po || do_fo) {
            T *gpo = do_po ? reinterpret_cast<T *>(args.out.partial_obs) + env0 * cfg.po_floats : nullptr;  // walked, not re-multiplied, per game
            T *gfo = do_fo ? reinterpret_cast<T *>(args.out.full_obs) + env0 * cfg.fo_floats : nullptr;
#pragma unroll 1
            for (int g = 0; g < toy::GAMES; g += NT) {
#pragma unroll
                for (int h = 0; h < NT; ++h) {  // NT tiles: one is patched while the others' copies are read
                    uint8_t *tile = tiles + h * tile_stride;
                    if (lane == 0) asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(NT - 1) : "memory");  // the copy NT games ago left this tile
                    __syncwarp();
                    if constexpr (half) {  // the tile at its row's residue mod 16: aligned body by TMA, head / tail by the lanes
                        T *tpo = reinterpret_cast<T *>(tile + ((h * po_bytes) & 15)), *tfo = reinterpret_cast<T *>(tile + po_slot + ((h * fo_bytes) & 15));
                        if (do_po) toy::restore_tile(cfg, tpo, pom, lane, undo_po[h]);
                        if (do_fo) toy::restore_tile(cfg, tfo, fom, lane, undo_fo[h]);
                        __syncwarp();
                        const uint8_t *st = stage + (g + h) * toy::STAGE_BYTES;
                        if (do_po) undo_po[h] = toy::patch_tile(cfg, st, tpo, pom, lane);
                        if (do_fo) undo_fo[h] = toy::patch_tile(cfg, st, tfo, fom, lane);
                        fence_async_smem();
                        __syncwarp();
                        if (do_po) emit_tile16<GT>(reinterpret_cast<uint8_t *>(gpo), reinterpret_cast<uint8_t *>(tpo), po_bytes);
                        if (do_fo) emit_tile16<GT>(reinterpret_cast<uint8_t *>(gfo), reinterpret_cast<uint8_t *>(tfo), fo_bytes);
                        if (lane == 0) bulk_commit();
                    } else {
                        if (do_po) toy::restore_tile(cfg, reinterpret_cast<float *>(tile), pom, lane, undo_po[h]);
                        if (do_fo) toy::restore_tile(cfg, reinterpret_cast<float *>(tile + po_bytes), fom, lane, undo_fo[h]);
                        __syncwarp();  // an entry being undone and a new entry of another lane may share an address
                        const uint8_t *st = stage + (g + h) * toy::STAGE_BYTES;
                        if (do_po) undo_po[h] = toy::patch_tile(cfg, st, reinterpret_cast<float *>(tile), pom, lane);
                        if (do_fo) undo_fo[h] = toy::patch_tile(cfg, st, reinterpret_cast<float *>(tile + po_bytes), fom, lane);
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            if (do_po) bulk_store(gpo, tile, uint32_t(po_bytes));
                            if (do_fo) bulk_store(gfo, tile + po_bytes, uint32_t(fo_bytes));
                            bulk_commit();
                        }
                    }
                    if (do_po) gpo += cfg.po_floats;
                    if (do_fo) gfo += cfg.fo_floats;
                }
            }
        }
    }
    if (do_tile && lane == 0) bulk_wait_read();  // shared memory must outlive the copies

    if (args.stats) {
        cnt.warp_sum();
        if (lane == 0) cnt.publish(args.stats);
    }
}

// ---- dense reference state <-> compact state (impl:16-60) -------------------------------------------
__global__ void sx_export_kernel(DevConfig cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
                                 long long num_envs, const int8_t *viewer, int64_t *dense, int8_t *player_out)
{
    const int lane = lane_id();
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= num_envs) return;
    const int N = cfg.N;
    // viewer -1: the state as that player sees it (impl:646-675): player layers swapped, board rotated 180 degrees
    const int flip = (viewer && viewer[env] == -1) ? 1 : 0;
    int64_t *d = dense + env * (long long)SX_NUM_STATE_LAYERS * N;
    for (int i = lane; i < SX_NUM_STATE_LAYERS * N; i += 32) d[i] = 0;
    __syncwarp();
    const uint4 aw = *reinterpret_cast<const uint4 *>(aux + env * 8);
    const uint32_t w[4] = {aw.x, aw.y, aw.z, aw.w};
    Aux a;
    aux_unpack(w, a);
    const uint8_t *b = board + env * cfg.board_stride;
    for (int p = lane; p < N; p += 32) {
        const uint32_t c = b[p];
        const int rank = c & CELL_RANK, owner = int((c >> 4) & 1) ^ flip, q = view(p, flip, N);
        if (c & CELL_OBST) d[2 * N + q] = 1;
        if (rank) {
            d[owner * N + q] = rank;
            d[(3 + owner) * N + q] = (c & CELL_REVEALED) ? rank : SP_UNKNOWN;
            if (c & CELL_STILL) d[(32 + owner) * N + q] = 1;
        }
    }
    if (lane == 0) {
        d[5 * N + 0] = a.turn;
        d[5 * N + 1] = a.over;
        d[5 * N + 2] = a.winner;
        d[5 * N + cfg.C + 0] = a.max_turns;
        d[5 * N + cfg.C + 1] = a.invalid;
        for (int s = 0; s < 2; ++s) {
            if (a.rfrom[s] != NO_CELL) d[(6 + (s ^ flip)) * N + view(a.rfrom[s], flip, N)] = 1;
            if (a.rto[s] != NO_CELL) d[(6 + (s ^ flip)) * N + view(a.rto[s], flip, N)] = -a.rcode[s];
        }
        if (player_out) player_out[env] = a.to_move == 0 ? 1 : -1;
    }
    const uint16_t *ce = cap + env * cfg.cap_stride;
    for (int e = lane; e < a.ncap; e += 32) {
        const uint32_t ent = ce[e];
        const int cell = ent & 0xff, owner = int((ent >> 8) & 1) ^ flip, type0 = (ent >> 9) & 15, count = int(ent >> 13) + 1;
        d[(8 + 12 * owner + type0) * N + view(cell, flip, N)] = count;
    }
}

__global__ void sx_import_kernel(DevConfig cfg, uint8_t *board, int16_t *aux, uint16_t *cap, long long num_envs,
                                 const int64_t *dense, const int8_t *player, uint8_t *status)
{
    const int lane = lane_id();
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= num_envs) return;
    const int N = cfg.N;
    const int64_t *d = dense + env * (long long)SX_NUM_STATE_LAYERS * N;
    uint8_t *b = board + env * cfg.board_stride;
    uint16_t *ce = cap + env * cfg.cap_stride;
    int err = 0;
    for (int p = lane; p < cfg.board_stride; p += 32) {
        uint32_t c = 0;
        if (p < N) {
            const int64_t t1 = d[p], t2 = d[N + p], ob = d[2 * N + p], po1 = d[3 * N + p], po2 = d[4 * N + p];
            const int64_t s1 = d[32 * N + p], s2 = d[33 * N + p];
            err |= (t1 < 0 || t1 > 12 || t2 < 0 || t2 > 12 || (t1 != 0 && t2 != 0));
            err |= (ob != 0 && ob != 1) || (s1 != 0 && s1 != 1) || (s2 != 0 && s2 != 1);
            err |= t1 ? (po1 != t1 && po1 != SP_UNKNOWN) : (po1 != 0);
            err |= t2 ? (po2 != t2 && po2 != SP_UNKNOWN) : (po2 != 0);
            err |= (s1 && !t1) || (s2 && !t2);
            if (ob) c |= CELL_OBST;
            if (t1) c |= uint32_t(t1) | (po1 == t1 ? CELL_REVEALED : 0) | (s1 ? CELL_STILL : 0);
            else if (t2) c |= uint32_t(t2) | CELL_OWNER | (po2 == t2 ? CELL_REVEALED : 0) | (s2 ? CELL_STILL : 0);
        }
        b[p] = uint8_t(c);
    }
    Aux a;
    for (int s = 0; s < 2; ++s) {
        int from = -1, to = -1, code = 0, nfrom = 0, nto = 0;
        for (int p = lane; p < N; p += 32) {
            const int64_t v = d[(6 + s) * N + p];
            if (v == 1) { from = p; nfrom++; }
            else if (v <= -1 && v >= -3) { to = p; code = int(-v); nto++; }
            else if (v != 0) err = 1;
        }
        for (int off = 16; off > 0; off >>= 1) {
            from = max(from, __shfl_xor_sync(FULL, from, off));
            to = max(to, __shfl_xor_sync(FULL, to, off));
            code = max(code, __shfl_xor_sync(FULL, code, off));
            nfrom += __shfl_xor_sync(FULL, nfrom, off);
            nto += __shfl_xor_sync(FULL, nto, off);
        }
        err |= nfrom > 1 || nto > 1;
        a.rfrom[s] = from < 0 ? NO_CELL : from;
        a.rto[s] = to < 0 ? NO_CELL : to;
        a.rcode[s] = to < 0 ? 0 : code;
    }
    int ncap = 0;
    for (int layer = 0; layer < 24; ++layer) {
        for (int p0 = 0; p0 < N; p0 += 32) {
            const int p = p0 + lane;
            int64_t cnt = 0;
            if (p < N) cnt = d[(8 + layer) * N + p];
            err |= cnt < 0 || cnt > SX_MAX_CAPTURE_COUNT;
            const bool has = cnt > 0 && cnt <= SX_MAX_CAPTURE_COUNT;
            const uint32_t vote = __ballot_sync(FULL, has);
            if (has) {
                const int slot = ncap + __popc(vote & ((1u << lane) - 1u));
                if (slot < cfg.cap_stride)
                    ce[slot] = uint16_t(cap_key(p, layer / 12, layer % 12 + 1) | (uint32_t(cnt - 1) << 13));
            }
            ncap += __popc(vote);
        }
    }
    err |= ncap > cfg.cap_stride;
    for (int e = ncap + lane; e < cfg.cap_stride; e += 32) ce[e] = 0;
    const int64_t turn = d[5 * N], over = d[5 * N + 1], winner = d[5 * N + 2], maxt = d[5 * N + cfg.C], inval = d[5 * N + cfg.C + 1];
    err |= turn < 0 || turn > 65535 || maxt < 0 || maxt > 65535 || (over != 0 && over != 1) || winner < -1 || winner > 1 ||
           (inval != 0 && inval != 1);
    err = __any_sync(FULL, err);
    a.turn = int(turn) & 0xffff;
    a.max_turns = int(maxt) & 0xffff;
    a.over = over != 0;
    a.invalid = inval != 0;
    a.winner = winner > 0 ? 1 : winner < 0 ? -1 : 0;
    a.to_move = (player && player[env] == -1) ? 1 : 0;
    a.ncap = min(ncap, cfg.cap_stride);
    a.overflow = 0;
    a.episode = 0;
    if (lane == 0) {
        uint32_t w[4];
        aux_pack(a, w);
        *reinterpret_cast<uint4 *>(aux + env * 8) = make_uint4(w[0], w[1], w[2], w[3]);
        if (status) status[env] = err ? 1 : 0;
    }
}

// uniform draw over the set entries of arbitrary uint8 masks (replaces maenv:830-834)
__global__ void sx_sample_kernel(const uint8_t *mask, long long num_envs, int mask_len, long long env_base, uint2 key,
                                 uint32_t step, int32_t *actions)
{
    const int lane = lane_id();
    const long long env = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= num_envs) return;
    const uint8_t *row = mask + env * mask_len;
    const int chunk = (mask_len + 31) / 32, lo = lane * chunk, hi = min(mask_len, lo + chunk);
    int mine = 0;
    for (int i = lo; i < hi; ++i) mine += row[i] != 0;
    int incl = mine;
    for (int off = 1; off < 32; off <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, off);
        if (lane >= off) incl += v;
    }
    const int total = __shfl_sync(FULL, incl, 31);
    const uint64_t gid = uint64_t(env_base + env);
    const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SAMPLE, step), key);
    int t = int(__umulhi(rnd.x, uint32_t(total)));
    int action = -1;
    const bool owner = total > 0 && t >= incl - mine && t < incl;
    if (owner) {
        t -= incl - mine;
        for (int i = lo; i < hi; ++i)
            if (row[i] != 0 && t-- == 0) { action = i; break; }
    }
    const uint32_t who = __ballot_sync(FULL, owner);
    action = who ? __shfl_sync(FULL, action, __ffs(who) - 1) : -1;
    if (lane == 0) actions[env] = action;
}

// impl:854-891: reward_matrix[rank the mover has on the start square][rank the opponent has on the end square] of the
// action each game is about to play; a no-op (and anything outside the action space) scores 0.  One thread per game.
__global__ void sx_heuristic_kernel(DevConfig cfg, const uint8_t *board, const int16_t *aux, long long num_envs,
                                    const int32_t *actions, int action_format, const float *matrix, float *rewards)
{
    const long long env = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (env >= num_envs) return;
    const uint4 aw = *reinterpret_cast<const uint4 *>(aux + env * 8);
    const uint32_t w[4] = {aw.x, aw.y, aw.z, aw.w};
    Aux a;
    aux_unpack(w, a);
    const int me = a.to_move;
    const Move mv = action_format == SX_ACTION_SPATIAL ? decode_spatial(cfg, actions[env], me) : decode_1d(cfg, actions[env]);
    float r = 0.0f;
    if (!mv.bad && !mv.noop) {
        const uint8_t *b = board + env * cfg.board_stride;
        const uint32_t sb = b[mv.start], eb = b[mv.end];
        const int own = int((sb >> 4) & 1) == me ? int(sb & CELL_RANK) : 0;      // owned_pieces[start], impl:879
        const int enemy = int((eb >> 4) & 1) != me ? int(eb & CELL_RANK) : 0;    // enemy_pieces[end], impl:880
        r = matrix[own * 13 + enemy];                                            // impl:882
    }
    rewards[env] = r;
}

}  // namespace sx

// =====================================================================================================
// host side
// =====================================================================================================
using namespace sx;

static thread_local std::string g_error;
static int fail(const std::string &msg)
{
    g_error = msg;
    return -1;
}
int sx_set_error(const std::string &msg) { return fail(msg); }  // for the other translation units of the library
static int cuda_fail(const char *what, cudaError_t e) { return fail(std::string(what) + ": " + cudaGetErrorString(e)); }

extern "C" const char *sx_last_error(void) { return g_error.c_str(); }
extern "C" int sx_version(void) { return 1; }

extern "C" int sx_config_create(const sx_config_desc *desc, sx_config **out)
{
    if (!desc || !out) return fail("sx_config_create: null argument");
    if (desc->rows < 3 || desc->cols < 3) return fail("Both rows and columns have to be at least 3");  // penv:28-30
    if (desc->rows > 15 || desc->cols > 15) return fail("boards larger than 15x15 are not supported");
    if (desc->max_turns < 1 || desc->max_turns > 65535) return fail("max_turns must be in 1..65535");
    if (!desc->obstacles || !desc->captured_lut || !desc->recent_lut || !desc->unit_lut) return fail("sx_config_create: null table");
    sx_config *c = new (std::nothrow) sx_config();
    if (!c) return fail("out of memory");
    DevConfig &d = c->dev;
    std::memset(&d, 0, sizeof(d));
    d.R = desc->rows; d.C = desc->cols; d.N = d.R * d.C;
    d.A = 2 * (d.R - 1) + 2 * (d.C - 1) + 1;
    d.mpa = d.R + d.C;
    d.magic_C = uint32_t((1ull << 32) / uint64_t(d.C)) + 1u;
    d.magic_A = uint32_t((1ull << 32) / uint64_t(d.A)) + 1u;
    d.magic_mpa = uint32_t((1ull << 32) / uint64_t(d.mpa)) + 1u;
    d.action_size = d.N * d.mpa + 1;
    d.board_stride = (d.N + 15) & ~15;
    d.max_turns = desc->max_turns;
    d.usable_rows = desc->usable_rows;
    d.setup_len = desc->usable_rows * d.C;
    d.p2_rot180 = desc->p2_rot180 ? 1 : 0;
    int pieces = 0;
    for (int t = 1; t <= 12; ++t) {
        if (desc->piece_amounts[t] < 0 || desc->piece_amounts[t] > SX_MAX_CAPTURE_COUNT) { delete c; return fail("piece amount out of range 0..8"); }
        for (int k = 0; k < desc->piece_amounts[t]; ++k) {
            if (pieces >= 128) { delete c; return fail("too many pieces"); }
            d.piece_seq[pieces++] = uint8_t(t);
        }
    }
    d.n_pieces = pieces;
    if (d.usable_rows < 1 || 2 * d.usable_rows > d.R || d.setup_len > 120 || pieces > d.setup_len) { delete c; return fail("pieces do not fit in the usable rows"); }
    if (desc->capture_capacity < 0 || desc->capture_capacity > 248) { delete c; return fail("capture_capacity out of range 0..248"); }
    d.cap_stride = std::max(8, ((desc->capture_capacity > 0 ? desc->capture_capacity : 2 * pieces) + 7) & ~7);
    d.original_channels = desc->obs_channel_mode == SX_CHANNELS_ORIGINAL ? 1 : 0;
    if (desc->obs_channel_mode != SX_CHANNELS_EXTENDED && desc->obs_channel_mode != SX_CHANNELS_ORIGINAL) { delete c; return fail("unknown obs_channel_mode"); }
    if (d.original_channels && (!desc->rank_lut || !desc->po_rank_lut)) { delete c; return fail("sx_config_create: the original channel mode needs rank_lut and po_rank_lut"); }
    d.po_ch = d.original_channels ? SX_PO_CHANNELS_ORIGINAL : SX_PO_CHANNELS;
    d.fo_ch = d.original_channels ? SX_FO_CHANNELS_ORIGINAL : SX_FO_CHANNELS;
    d.po_floats = d.N * d.po_ch;
    d.fo_floats = d.N * d.fo_ch;
    if (d.original_channels) {
        std::memcpy(d.rank_lut, desc->rank_lut, sizeof(d.rank_lut));
        std::memcpy(d.po_rank_lut, desc->po_rank_lut, sizeof(d.po_rank_lut));
    }
    d.mask_bytes = d.N * d.A;
    std::memcpy(d.cap_lut, desc->captured_lut, sizeof(d.cap_lut));
    std::memcpy(d.recent_lut, desc->recent_lut, sizeof(d.recent_lut));
    std::memcpy(d.unit_lut, desc->unit_lut, sizeof(d.unit_lut));
    if (desc->obs_dtype != SX_DTYPE_F32 && desc->obs_dtype != SX_DTYPE_BF16 && desc->obs_dtype != SX_DTYPE_F16) {
        delete c;
        return fail("sx_config_create: obs_dtype must be SX_DTYPE_F32 (0), SX_DTYPE_BF16 (1) or SX_DTYPE_F16 (2)");
    }
    c->obs_elem_bytes = desc->obs_dtype == SX_DTYPE_F32 ? 4 : 2;
    if (c->obs_elem_bytes == 2) {
        // 16-bit observations: every LUT word becomes the round-to-nearest-even bit pattern in its low half (obs_value),
        // so the kernels only store 16-bit words and bfloat16 / float16 share one code path
        const bool bf16 = desc->obs_dtype == SX_DTYPE_BF16;
        auto to16 = [bf16](float &v) {
            uint32_t bits;
            if (bf16) { const __nv_bfloat16_raw r = __float2bfloat16_rn(v); bits = r.x; }
            else { const __half_raw r = __float2half_rn(v); bits = r.x; }
            std::memcpy(&v, &bits, sizeof(v));
        };
        for (float &v : d.cap_lut) to16(v);
        for (float &v : d.recent_lut) to16(v);
        for (float &v : d.unit_lut) to16(v);
        for (float &v : d.rank_lut) to16(v);
        for (float &v : d.po_rank_lut) to16(v);
    }
    for (int i = 0; i < d.N; ++i) d.obstacles[i] = desc->obstacles[i] ? 1 : 0;
    // games per warp: small boards share a warp (each game needs max(R, C) <= lanes / 2 and N <= 2 * lanes)
    const int side = std::max(d.R, d.C);
    c->games_per_warp = (side <= 4 && d.N <= 16) ? 4 : (side <= 8 && d.N <= 32) ? 2 : 1;
    const int lanes = 32 / c->games_per_warp;
    const int k = (d.N + lanes - 1) / lanes;
    c->cells_per_lane = k <= 2 ? 2 : k <= 4 ? 4 : 8;
    // dense boards of the 10x10 class: movers are handed to lanes (measured: Standard, 40 pieces a side, +4 %; Barrage, 8
    // pieces, -3 %; profiles/r3g_all_boards.txt)
    c->compact_movers = c->cells_per_lane == 4 && c->games_per_warp == 1 && pieces > 16;
    sx_layout &l = c->layout;
    l.rows = d.R; l.cols = d.C; l.cells = d.N; l.spatial_channels = d.A; l.spatial_actions = d.mask_bytes;
    l.action_size = d.action_size; l.board_stride = d.board_stride; l.aux_stride = 8; l.captured_stride = d.cap_stride;
    l.po_floats = d.po_floats; l.fo_floats = d.fo_floats; l.setup_len = d.setup_len; l.pieces_per_side = pieces;
    l.po_channels = d.po_ch; l.fo_channels = d.fo_ch;
    l.obs_elem_bytes = c->obs_elem_bytes;
    *out = c;
    return 0;
}

extern "C" void sx_config_destroy(sx_config *cfg) { delete cfg; }

extern "C" int sx_config_set_start_states(sx_config *cfg, sx_state table, int64_t n_states, int32_t *start_index_d,
                                          int64_t index_env_base, int64_t index_len)
{
    if (!cfg) return fail("sx_config_set_start_states: null config");
    if (n_states < 0 || n_states > 0x7fffffffLL) return fail("sx_config_set_start_states: n_states out of range");
    if (n_states > 0 && table.board != nullptr && (!table.aux || !table.captured))
        return fail("sx_config_set_start_states: the table needs board, aux and captured tensors");
    const bool on = n_states > 0 && table.board != nullptr;
    cfg->start_states = on ? table : sx_state{nullptr, nullptr, nullptr};
    cfg->n_start_states = on ? n_states : 0;
    cfg->start_index = (on && index_len > 0) ? start_index_d : nullptr;
    cfg->start_index_base = index_env_base;
    cfg->start_index_len = cfg->start_index ? index_len : 0;
    return 0;
}

// Result-preserving launch tuning (include/stratego_b200.h): lets tools/sweep_tuning.py time the shipped library under
// other launch shapes than the built-in ones.  None of the three settings changes a result.
extern "C" int sx_config_set_tuning(sx_config *cfg, int32_t warps_per_block, int32_t issue_point, int32_t compact_movers)
{
    if (!cfg) return fail("sx_config_set_tuning: null config");
    if (warps_per_block > 32 || issue_point > 2) return fail("sx_config_set_tuning: warps_per_block <= 32, issue_point 0..2");
    {
        std::lock_guard<std::mutex> lock(cfg->plan_mutex);
        cfg->plans.clear();  // launch shapes are cached per configuration
    }
    if (warps_per_block >= 0) cfg->tune_warps = warps_per_block;
    if (issue_point >= 0) cfg->tune_issue = issue_point;
    if (compact_movers >= 0) {
        cfg->compact_movers = compact_movers != 0 && cfg->cells_per_lane == 4 && cfg->games_per_warp == 1;
        cfg->compact_forced = true;
    }
    return 0;
}

extern "C" int sx_config_layout(const sx_config *cfg, sx_layout *out)
{
    if (!cfg || !out) return fail("sx_config_layout: null argument");
    *out = cfg->layout;
    return 0;
}

typedef void (*fused_fn)(const KernelArgs);
// the modes without observations (lean step, mask only) share the float instantiation whatever the element type
template <int K, int G, bool CM, class T>
static fused_fn fused_for_mode_typed(int mode)
{
    switch (mode) {
    case MODE_STEP_PO_MASK: return sx_fused_kernel<K, MODE_STEP_PO_MASK, G, CM, T>;
    case MODE_STEP_PO_FO_MASK: return sx_fused_kernel<K, MODE_STEP_PO_FO_MASK, G, CM, T>;
    case MODE_STEP_LEAN: return sx_fused_kernel<K, MODE_STEP_LEAN, G, CM>;
    case MODE_MASK: return sx_fused_kernel<K, MODE_MASK, G, CM>;
    case MODE_OBSERVE_PO_MASK: return sx_fused_kernel<K, MODE_OBSERVE_PO_MASK, G, CM, T>;
    default: return sx_fused_kernel<K, MODE_GENERIC, G, CM, T>;
    }
}
template <int K, int G, bool CM = false>
static fused_fn fused_for_mode(int mode, int obs_elem_bytes)
{
    return obs_elem_bytes == 2 ? fused_for_mode_typed<K, G, CM, uint16_t>(mode) : fused_for_mode_typed<K, G, CM, float>(mode);
}
// (cells per lane, games per warp) instantiations: (2,4) boards up to 4x4, (2,2) up to 5x5 (both dimensions must fit
// in half a group's lanes), (2,1) up to 64 cells, (4,1) 10x10, (8,1) 15x15
static fused_fn fused_for(const sx_config *cfg, int mode)
{
    const int k = cfg->cells_per_lane, g = cfg->games_per_warp, eb = cfg->obs_elem_bytes;
    if (g == 4) return fused_for_mode<2, 4>(mode, eb);
    if (g == 2) return fused_for_mode<2, 2>(mode, eb);
    switch (k) {
    case 2: return fused_for_mode<2, 1>(mode, eb);
    case 4: {
        // measured on the shipped library (profiles/r3o_shipped_tuning_sweep.txt): Standard with one observation 169.0 ->
        // 176.0 M env-steps/s with compact movers, with both observations 89.9 -> 88.1 M (6 warps per SM there)
        // (observe-only launches: 0.730 -> 0.753 ms per 131 072 Standard games; mask-only 0.252 -> 0.201 ms, lean step 0.243
        // -> 0.188 ms, profiles/r3p_all_boards.txt)
        const bool compact = cfg->compact_movers &&
                             (cfg->compact_forced || (mode != MODE_STEP_PO_FO_MASK && mode != MODE_OBSERVE_PO_MASK));
        return compact ? fused_for_mode<4, 1, true>(mode, eb) : fused_for_mode<4, 1>(mode, eb);
    }
    default: return fused_for_mode<8, 1>(mode, eb);
    }
}

// the specialised kernel for this launch, if one matches exactly
static int mode_for(const sx_config *cfg, const KernelArgs &a)
{
    if (a.reset_mask || a.setup_idx || a.mask1d) return MODE_GENERIC;
    if (cfg->dev.original_channels && (a.ops & (OP_PO | OP_FO))) return MODE_GENERIC;
    for (int mode : {MODE_MASK, MODE_OBSERVE_PO_MASK})
        if (a.ops == mode_ops(mode) && !(a.flags & SX_SAMPLE_NEXT)) return mode;
    if (a.player_override) return MODE_GENERIC;
    for (int mode : {MODE_STEP_PO_MASK, MODE_STEP_PO_FO_MASK, MODE_STEP_LEAN})
        if (a.ops == mode_ops(mode)) return mode;
    return MODE_GENERIC;
}



// Launch shape of the 16-bit observations, per board class: resident warps per SM and where a stepping game's
// background copy is issued (0 late, 1 after the outcome, 2 top of the game; sx_fused_kernel).  Half the bytes per game
// move the optimum of the float32 rule ("~230 KB in flight per SM", plan_launch_uncached), so these come from their own
// sweep (tools/bench_obs_dtype.py --sweep, profiles/r5a_obs_dtype_sweep.txt; B200 at 1 000 W).  16 warps is the most
// the 128-register kernels keep resident.  Barrage bf16: 10 warps (the float32 rule) 1.226 ms, 12: 1.057, 16: 0.895 ms;
// Standard 2.523 / 2.213 / 2.056 ms; Standard PO + full 10: 1.917, 12: 1.851, 16: 1.966 ms; 8x8 16 warps 1.414 ms
// (12: 1.674); issue point 1 is best or within 0.5 % everywhere but on 15x15 (late 1.268, 1: 1.276 ms).
struct Shape16 {
    int warps, issue;
};
static Shape16 shape16(const DevConfig &d, uint32_t ops)
{
    const bool both = (ops & OP_PO) && (ops & OP_FO);
    if (d.N > 128) return {both ? 10 : 16, 0};  // 15x15 (both observations not swept: the float32 choice)
    if (d.N >= 100) return {both ? 12 : 16, 1};  // 10x10
    return {16, 1};                              // 8x8, 6x6, 5x5 and the warp-level path of the toy boards
}

// Block shape: one block per SM with as many warps as the register file allows
// (sx_config_set_tuning overrides); the block's shared memory is the background images plus one small slice per warp.
static int plan_launch_uncached(const sx_config *cfg, uint32_t ops, int mode, long long num_envs, LaunchPlan *plan,
                                int compressed_warps);

// Launch shape of a 10x10 float32 step whose observation / mask planes all lie in compressible memory (sx_device_alloc),
// 0 for any other launch.  The memory system then writes fewer DRAM bytes, DRAM stops limiting the write stream, and
// more copies in flight pay off (tools/sweep_tuning.py on compressible outputs, profiles/r4c_compressed_shape_sweep.txt;
// env-steps/s at the plain shape -> here): one observation + mask 12 warps with the copy issued late, Barrage 188.4 M ->
// 217.3 M, Standard 179.2 M -> 196.7 M; both observations 7 warps, late, 91.1 M -> 99.1 M.  Every shape gives the same
// results (tests/test_tuning_gpu.py).
static int compressed_shape_warps(const sx_config *cfg, uint32_t ops)
{
    if (cfg->obs_elem_bytes != 4 || !(ops & OP_STEP) || !(ops & (OP_PO | OP_FO)) || cfg->dev.N < 100 || cfg->dev.N > 128)
        return 0;
    return (ops & OP_PO) && (ops & OP_FO) ? 7 : 12;
}

static bool outputs_compressible(const sx_outputs &out)
{
    for (const void *p : {static_cast<const void *>(out.partial_obs), static_cast<const void *>(out.full_obs),
                          static_cast<const void *>(out.valid_mask)})
        if (p && !sx_in_compressible_allocation(p)) return false;
    return true;
}

static int compressed_warps_for(const sx_config *cfg, const sx_outputs &out, uint32_t ops)
{
    const int w = compressed_shape_warps(cfg, ops);
    return w && outputs_compressible(out) ? w : 0;
}

static int plan_launch(const sx_config *cfg, uint32_t ops, int mode, long long num_envs, LaunchPlan *plan,
                       int compressed_warps = 0)
{
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return cuda_fail("cudaGetDevice", e);
    const uint64_t key = (uint64_t(uint32_t(device)) << 40) | (uint64_t(compressed_warps) << 24) | (uint64_t(ops) << 8) |
                         uint64_t(mode);
    {
        std::lock_guard<std::mutex> lock(cfg->plan_mutex);
        auto it = cfg->plans.find(key);
        if (it == cfg->plans.end()) {
            LaunchPlan full;
            if (int rc = plan_launch_uncached(cfg, ops, mode, 1LL << 40, &full, compressed_warps)) return rc;
            it = cfg->plans.emplace(key, full).first;
        }
        *plan = it->second;
    }
    const long long per_block = (long long)plan->warps_per_block * cfg->games_per_warp;
    const long long needed = (num_envs + per_block - 1) / per_block;
    plan->grid = int(std::max(1LL, std::min((long long)plan->num_sms * plan->blocks_per_sm, needed)));
    return 0;
}

static int tile_bytes_for(const sx_config *cfg, uint32_t ops)
{
    return cfg->obs_elem_bytes == 2 ? carve_tile<2>(cfg->dev, ops, nullptr, nullptr) : carve_tile<4>(cfg->dev, ops, nullptr, nullptr);
}

static int plan_launch_uncached(const sx_config *cfg, uint32_t ops, int mode, long long num_envs, LaunchPlan *plan,
                                int compressed_warps)
{
    const int warp_bytes = carve_warp(cfg->dev, nullptr, nullptr);
    const int tile_bytes = tile_bytes_for(cfg, ops);
    fused_fn fn = fused_for(cfg, mode);
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return cuda_fail("cudaGetDevice", e);
    int num_sms = 0, max_smem_optin = 0;
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin);
    if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute", e);
    cudaFuncAttributes attr;
    e = cudaFuncGetAttributes(&attr, fn);
    if (e != cudaSuccess) return cuda_fail("cudaFuncGetAttributes", e);
    const int max_warps = std::max(1, std::min(attr.maxThreadsPerBlock / 32, 32));
    // Measured on B200: throughput peaks when ~0.4 MB of output per SM is in flight and falls beyond it (more
    // resident warps only lengthen the TMA completion queue), so fewer warps for bigger per-game outputs.
    // 8 warps is a sharp optimum for one 10x10 observation + mask (7: -11 %, 9 and more: -3 to -12 %, not monotonic).
    // Smaller boards carry less output per game, so more of them fit in the same bytes in flight: 8x8 (19 KB per game)
    // 10 warps 218 M, 12 warps 237 M, 16 warps 255 M env-steps/s with the copy issued late.
    // 6x6 (10.4 KB per game): 10 warps 234 M, 16 warps 324 M, 24 warps 363 M, 32 warps 330 M (all with the 64-register
    // build of round 1).  Rule for boards below 10x10: about 230 KB of output in flight per SM -- the same figure that
    // makes 8 warps the optimum of the 10x10 boards; with 128 registers per thread (no spills) the 8x8 board peaks at
    // 12 warps (272 M env-steps/s; 16 warps 256 M) and the 6x6 board at the 16 warps that fit (372 M).
    const int small_board = std::max(8, std::min(32, (232 * 1024 + tile_bytes / 2) / std::max(1, tile_bytes)));
    int preferred = tile_bytes <= 8 * 1024 ? 32 : tile_bytes <= 32 * 1024 ? (cfg->dev.N >= 100 ? 8 : small_board)
                    : tile_bytes <= 64 * 1024 ? 6 : 10;  // 15x15 (74 KB per game): 4 warps 39 M, 6: 55 M, 8: 69 M, 10: 75 M env-steps/s
    if (cfg->obs_elem_bytes == 2 && (ops & (OP_PO | OP_FO))) preferred = shape16(cfg->dev, ops).warps;
    if (compressed_warps) preferred = compressed_warps;
    int warps = std::min(max_warps, std::max(1, cfg->tune_warps > 0 ? cfg->tune_warps : preferred));
    const int games = cfg->games_per_warp;  // each game of a warp has its own slice
    while (warps > 1 && tile_bytes + warps * games * warp_bytes > max_smem_optin) --warps;
    const int smem = tile_bytes + warps * games * warp_bytes;
    if (smem > max_smem_optin) return fail("variant does not fit in shared memory");
    int blocks = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, fn, warps * 32, size_t(smem));
    if (e != cudaSuccess) return cuda_fail("cudaOccupancyMaxActiveBlocksPerMultiprocessor", e);
    if (blocks < 1) return fail("fused kernel cannot be resident on this device");
    if (tile_bytes > 8 * 1024) blocks = 1;
    plan->warps_per_block = warps;
    plan->blocks_per_sm = blocks;
    plan->smem_per_block = smem;
    plan->num_sms = num_sms;
    plan->regs = attr.numRegs;
    plan->warp_bytes = warp_bytes;
    plan->tile_bytes = tile_bytes;
    const long long grid = (long long)num_sms * blocks;
    const long long needed = (num_envs + warps * games - 1) / (warps * games);
    plan->grid = int(std::max(1LL, std::min(grid, needed)));
    return 0;
}


// ---- toy-board launch (sx_toy_kernel) ------------------------------------------------------------------------------------
// Eligible: at most 16 cells with 16-byte aligned observation rows, a board / capture list of 16 bytes each, at most 8
// setup cells and pieces, extended channels, and one of the three step modes without per-launch overrides.
static bool toy_eligible(const sx_config *cfg, const KernelArgs &a, int mode)
{
    const DevConfig &d = cfg->dev;
    if (a.flags & (SX_KERNEL_BASELINE | SX_REPEAT_OTHER_SIDE)) return false;
    if (a.out.terminal_partial_obs || a.out.terminal_full_obs) return false;
    if (cfg->n_start_states > 0) return false;  // curriculum starts are a warp-level kernel feature
    if (mode != MODE_STEP_PO_MASK && mode != MODE_STEP_PO_FO_MASK && mode != MODE_STEP_LEAN) return false;
    if (d.N > 16 || (d.N & 3) != 0 || d.A > 16 || d.board_stride != 16 || d.cap_stride != 8) return false;
    if (d.setup_len > 8 || d.n_pieces > 8 || d.original_channels) return false;
    if (a.player_override || a.reset_mask || a.setup_idx || a.mask1d) return false;
    // the kernel moves state as 16-byte words and observations as bulk copies: everything must be 16-byte aligned
    // (torch / cudaMalloc allocations and whole-game offsets into them always are)
    const uintptr_t bits = reinterpret_cast<uintptr_t>(a.board) | reinterpret_cast<uintptr_t>(a.aux) |
                           reinterpret_cast<uintptr_t>(a.cap) | reinterpret_cast<uintptr_t>(a.out.partial_obs) |
                           reinterpret_cast<uintptr_t>(a.out.full_obs);
    if (bits & 15) return false;
    return a.num_envs >= toy::GAMES;
}

typedef void (*toy_fn)(const KernelArgs);
static toy_fn toy_for_mode(int mode, int obs_elem_bytes)
{
    if (obs_elem_bytes == 2 && mode != MODE_STEP_LEAN)
        return mode == MODE_STEP_PO_MASK ? sx_toy_kernel<MODE_STEP_PO_MASK, uint16_t> : sx_toy_kernel<MODE_STEP_PO_FO_MASK, uint16_t>;
    return mode == MODE_STEP_PO_MASK ? sx_toy_kernel<MODE_STEP_PO_MASK>
         : mode == MODE_STEP_PO_FO_MASK ? sx_toy_kernel<MODE_STEP_PO_FO_MASK> : sx_toy_kernel<MODE_STEP_LEAN>;
}

// host mirror of the shared-memory slice of one warp of sx_toy_kernel
static int toy_warp_bytes(const sx_config *cfg, uint32_t ops)
{
    const DevConfig &d = cfg->dev;
    const int eb = cfg->obs_elem_bytes;
    const int mask_img = (ops & OP_MASK) ? round16(toy::GAMES * d.mask_bytes + 16) : 0;
    const int po = (ops & OP_PO) ? d.po_floats * eb : 0, fo = (ops & OP_FO) ? d.fo_floats * eb : 0;
    const int tile = eb == 2 ? toy::tile_slot(po) + toy::tile_slot(fo) : po + fo;
    return toy::GAMES * toy::STAGE_BYTES + mask_img + TOY_TILES * tile;
}

struct ToyPlan {
    int warps, smem, grid_max, tile_bytes, warp_bytes, num_sms;
};
static int plan_toy(const sx_config *cfg, uint32_t ops, ToyPlan *plan)
{
    int device = 0, max_smem = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return cuda_fail("cudaGetDevice", e);
    cudaDeviceGetAttribute(&plan->num_sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    plan->tile_bytes = tile_bytes_for(cfg, ops);
    plan->warp_bytes = toy_warp_bytes(cfg, ops);
    // 12 warps per SM (or as many as shared memory holds): Micro 8 warps 1.10 G, 10: 1.35 G, 11: 1.42 G, 12: 1.49 G,
    // 13-16: 1.40-1.43 G env-steps/s; Tiny 8: 1.02 G, 10-13: 1.08 G
    // (Tiny 4x4 peaks at 11 warps: 1 113 M vs 1 072 M at 12, measured twice, profiles/r2o_*, r2t_*.  A warp sync between a
    // pass's commit_group and the next pass's wait_group.read changes nothing here: that wait is for an older group.)
    plan->warps = std::min(TOY_THREADS / 32, cfg->dev.N <= 12 ? 12 : 11);
    while (plan->warps > 1 && plan->tile_bytes + plan->warps * plan->warp_bytes > max_smem) --plan->warps;
    plan->smem = plan->tile_bytes + plan->warps * plan->warp_bytes;
    if (plan->smem > max_smem) return fail("toy kernel does not fit in shared memory");
    plan->grid_max = plan->num_sms;
    return 0;
}

static int launch_toy(const sx_config *cfg, KernelArgs &args, int mode, cudaStream_t stream)
{
    const uint32_t ops = mode_ops(mode);
    ToyPlan plan;
    if (int rc = plan_toy(cfg, ops, &plan)) return rc;
    toy_fn fn = toy_for_mode(mode, cfg->obs_elem_bytes);
    static std::mutex attr_mutex;
    {
        std::lock_guard<std::mutex> lock(attr_mutex);
        cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, plan.smem);
        if (e != cudaSuccess) return cuda_fail("cudaFuncSetAttribute", e);
    }
    args.cfg = cfg->dev;
    args.ops = ops;
    args.warp_bytes = plan.warp_bytes;
    args.tile_bytes = plan.tile_bytes;
    const long long groups = args.num_envs / toy::GAMES;
    const int grid = int(std::max(1LL, std::min((long long)plan.grid_max, (groups + plan.warps - 1) / plan.warps)));
    fn<<<grid, plan.warps * 32, plan.smem, stream>>>(args);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail("sx toy kernel launch", e);
}

// `elems` observation elements of the configuration's type past p
static float *obs_at(const sx_config *cfg, float *p, int64_t elems)
{
    return p ? reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(p) + elems * cfg->obs_elem_bytes) : nullptr;
}

// the outputs of the games from `lo` on
static sx_outputs offset_outputs(const sx_config *cfg, const sx_outputs &o, int64_t lo)
{
    const DevConfig &d = cfg->dev;
    sx_outputs r = o;
    r.partial_obs = obs_at(cfg, r.partial_obs, lo * d.po_floats);
    r.full_obs = obs_at(cfg, r.full_obs, lo * d.fo_floats);
    if (r.valid_mask) r.valid_mask += lo * d.mask_bytes;
    if (r.reward) r.reward += lo;
    if (r.done) r.done += lo;
    if (r.winner) r.winner += lo;
    if (r.ending_invalid) r.ending_invalid += lo;
    if (r.illegal) r.illegal += lo;
    if (r.player) r.player += lo;
    if (r.next_action) r.next_action += lo;
    r.terminal_partial_obs = obs_at(cfg, r.terminal_partial_obs, lo * 2 * d.po_floats);
    r.terminal_full_obs = obs_at(cfg, r.terminal_full_obs, lo * 2 * d.fo_floats);
    return r;
}

static int launch_fused(const sx_config *cfg, KernelArgs &args, cudaStream_t stream)
{
    if (args.num_envs <= 0) return 0;
    args.start_board = cfg->start_states.board; args.start_aux = cfg->start_states.aux; args.start_cap = cfg->start_states.captured;
    args.n_start = cfg->start_states.board ? uint32_t(cfg->n_start_states) : 0u;
    args.start_index = cfg->start_index; args.start_index_base = cfg->start_index_base; args.start_index_len = cfg->start_index_len;
    LaunchPlan plan;
    const int mode = mode_for(cfg, args);
    if (toy_eligible(cfg, args, mode)) {
        // whole groups of 32 games go to the thread-per-game kernel, the last num_envs % 32 games to the warp-level one
        const long long whole = args.num_envs / toy::GAMES * toy::GAMES, rest = args.num_envs - whole;
        KernelArgs head = args;
        head.num_envs = whole;
        if (int rc = launch_toy(cfg, head, mode, stream)) return rc;
        if (rest == 0) return 0;
        args.board += whole * cfg->dev.board_stride;
        args.aux += whole * 8;
        args.cap += whole * cfg->dev.cap_stride;
        args.actions += whole;
        args.env_base += whole;
        args.num_envs = rest;
        args.out = offset_outputs(cfg, args.out, whole);
    }
    if (int rc = plan_launch(cfg, args.ops, mode, args.num_envs, &plan, compressed_warps_for(cfg, args.out, args.ops))) return rc;
    args.cfg = cfg->dev;
    args.warp_bytes = plan.warp_bytes;
    args.tile_bytes = plan.tile_bytes;
    // launches without a step (sx_observe, sx_valid_mask, the observe pass of a reset) issue their copies late
    if (!(args.ops & OP_STEP)) args.flags |= SX_TUNE_COMMIT_GAP;
    // (Tried and removed: marking the state range as persisting in L2 with an access-policy window.  A pure store
    // stream loses ~8 % when the ~0.2 KB/game state reads come from DRAM (tools/probes/probe_write.cu), but any L2
    // set-aside large enough to hold the state takes capacity from the output lines that wait for their sparse
    // stores: 25-30 % of the maximum was neutral, 35 % and more cost 15-35 %.)
    fused_for(cfg, mode)<<<plan.grid, plan.warps_per_block * 32, plan.smem_per_block, stream>>>(args);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail("sx fused kernel launch", e);
    return 0;
}

static uint2 make_key(uint64_t seed) { return make_uint2(uint32_t(seed), uint32_t(seed >> 32)); }

static void base_args(KernelArgs &a, sx_state st, int64_t num_envs, int64_t env_base)
{
    std::memset(&a, 0, sizeof(a));
    a.board = st.board; a.aux = st.aux; a.cap = st.captured;
    a.num_envs = num_envs; a.env_base = env_base;
}

static int check_state(const sx_config *cfg, sx_state st, const char *who)
{
    if (!cfg) return fail(std::string(who) + ": null config");
    if (!st.board || !st.aux || !st.captured) return fail(std::string(who) + ": null state tensor");
    return 0;
}

extern "C" int sx_reset(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const uint8_t *reset_mask_d,
                        const uint8_t *setups_d, int32_t n_setups, const int32_t *setup_idx_d, uint64_t seed, uint32_t flags,
                        void *stream)
{
    if (int rc = check_state(cfg, st, "sx_reset")) return rc;
    if (!(flags & SX_RESET_RANDOM_SHUFFLE) && (!setups_d || n_setups < 1) && cfg->n_start_states == 0)
        return fail("sx_reset: a setup table or SX_RESET_RANDOM_SHUFFLE is required");
    KernelArgs a;
    base_args(a, st, num_envs, env_base);
    a.ops = OP_RESET | OP_WRITE_STATE;
    a.flags = flags & (SX_RESET_RANDOM_SHUFFLE | SX_SAME_SETUP | SX_REPEAT_OTHER_SIDE);
    a.setups = setups_d; a.n_setups = n_setups; a.setup_idx = setup_idx_d; a.reset_mask = reset_mask_d;
    a.key = make_key(seed);
    return launch_fused(cfg, a, static_cast<cudaStream_t>(stream));
}

extern "C" int sx_import_ref_state(const sx_config *cfg, sx_state st, int64_t num_envs, const int64_t *dense_d,
                                   const int8_t *player_d, uint8_t *status_d, void *stream)
{
    if (int rc = check_state(cfg, st, "sx_import_ref_state")) return rc;
    if (!dense_d) return fail("sx_import_ref_state: null dense state");
    if (num_envs <= 0) return 0;
    const int wpb = 4;
    sx_import_kernel<<<unsigned((num_envs + wpb - 1) / wpb), wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        cfg->dev, st.board, st.aux, st.captured, num_envs, dense_d, player_d, status_d);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail("sx_import_kernel", e);
}

static int export_impl(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *viewer_d, int64_t *dense_d,
                       int8_t *player_d, void *stream, const char *who)
{
    if (int rc = check_state(cfg, st, who)) return rc;
    if (!dense_d) return fail(std::string(who) + ": null dense state");
    if (num_envs <= 0) return 0;
    const int wpb = 4;
    sx_export_kernel<<<unsigned((num_envs + wpb - 1) / wpb), wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        cfg->dev, st.board, st.aux, st.captured, num_envs, viewer_d, dense_d, player_d);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail("sx_export_kernel", e);
}

extern "C" int sx_export_ref_state(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t *dense_d, int8_t *player_d,
                                   void *stream)
{
    return export_impl(cfg, st, num_envs, nullptr, dense_d, player_d, stream, "sx_export_ref_state");
}

extern "C" int sx_export_perspective_state(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *viewer_d,
                                           int64_t *dense_d, void *stream)
{
    return export_impl(cfg, st, num_envs, viewer_d, dense_d, nullptr, stream, "sx_export_perspective_state");
}

extern "C" int sx_valid_mask(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *player_d, int32_t format,
                             uint8_t *mask_d, void *stream)
{
    if (int rc = check_state(cfg, st, "sx_valid_mask")) return rc;
    if (!mask_d) return fail("sx_valid_mask: null output");
    KernelArgs a;
    base_args(a, st, num_envs, 0);
    a.player_override = player_d;
    if (format == SX_ACTION_SPATIAL) {
        a.ops = OP_MASK;
        a.out.valid_mask = mask_d;
    } else if (format == SX_ACTION_1D) {
        cudaError_t e = cudaMemsetAsync(mask_d, 0, size_t(num_envs) * cfg->dev.action_size, static_cast<cudaStream_t>(stream));
        if (e != cudaSuccess) return cuda_fail("cudaMemsetAsync", e);
        a.ops = OP_MASK_1D;
        a.mask1d = mask_d;
    } else {
        return fail("sx_valid_mask: unknown format");
    }
    return launch_fused(cfg, a, static_cast<cudaStream_t>(stream));
}

extern "C" int sx_observe(const sx_config *cfg, sx_state st, int64_t num_envs, const int8_t *player_d, sx_outputs out,
                          void *stream)
{
    if (int rc = check_state(cfg, st, "sx_observe")) return rc;
    KernelArgs a;
    base_args(a, st, num_envs, 0);
    a.player_override = player_d;
    a.out = out;
    a.out.next_action = nullptr;
    a.ops = (out.valid_mask ? OP_MASK : 0) | (out.partial_obs ? OP_PO : 0) | (out.full_obs ? OP_FO : 0);
    if (a.ops == 0 && !out.player) return 0;
    return launch_fused(cfg, a, static_cast<cudaStream_t>(stream));
}

extern "C" int sx_step(const sx_config *cfg, sx_state st, int64_t num_envs, const int32_t *actions_d, int32_t action_format,
                       uint32_t flags, sx_outputs out, void *stream)
{
    if (int rc = check_state(cfg, st, "sx_step")) return rc;
    if (!actions_d) return fail("sx_step: null actions");
    if (action_format != SX_ACTION_SPATIAL && action_format != SX_ACTION_1D) return fail("sx_step: unknown action format");
    KernelArgs a;
    base_args(a, st, num_envs, 0);
    a.actions = actions_d; a.action_format = action_format;
    a.flags = flags & SX_ALLOW_OSCILLATION;
    a.out = out;
    a.out.partial_obs = nullptr; a.out.full_obs = nullptr; a.out.valid_mask = nullptr; a.out.next_action = nullptr;
    a.out.terminal_partial_obs = nullptr; a.out.terminal_full_obs = nullptr;
    a.ops = OP_STEP | OP_WRITE_STATE | OP_NEED_MOVES;
    return launch_fused(cfg, a, static_cast<cudaStream_t>(stream));
}

static uint32_t step_all_ops(const sx_outputs &out)
{
    uint32_t ops = OP_STEP | OP_WRITE_STATE | OP_NEED_MOVES;
    if (out.valid_mask) ops |= OP_MASK;
    if (out.partial_obs) ops |= OP_PO;
    if (out.full_obs) ops |= OP_FO;
    return ops;
}

extern "C" int sx_step_all(const sx_config *cfg, sx_state st, int64_t num_envs, int64_t env_base, const int32_t *actions_d,
                           int32_t action_format, uint32_t flags, const uint8_t *setups_d, int32_t n_setups, uint64_t seed,
                           sx_outputs out, int64_t *stats_d, void *stream)
{
    if (int rc = check_state(cfg, st, "sx_step_all")) return rc;
    if (!actions_d) return fail("sx_step_all: null actions");
    if (action_format != SX_ACTION_SPATIAL && action_format != SX_ACTION_1D) return fail("sx_step_all: unknown action format");
    if ((flags & SX_AUTO_RESET) && !(flags & SX_RESET_RANDOM_SHUFFLE) && (!setups_d || n_setups < 1) && cfg->n_start_states == 0)
        return fail("sx_step_all: auto-reset needs a setup table or SX_RESET_RANDOM_SHUFFLE");
    if ((out.terminal_partial_obs && !out.partial_obs) || (out.terminal_full_obs && !out.full_obs))
        return fail("sx_step_all: a terminal observation buffer needs its regular observation output in the same call");
    KernelArgs a;
    base_args(a, st, num_envs, env_base);
    a.actions = actions_d; a.action_format = action_format;
    // flag bits 20-21: where a game's background copy is issued (0 late, 1 after the outcome, 2 top of the game).
    // B200 sweeps (profiles/r1k_sweeps.txt): a 10x10 board with ONE observation is fastest with the copy issued after the
    // outcome at 8 warps per SM; both observations and the smaller boards issue late.
    const bool one_obs = (out.partial_obs != nullptr) != (out.full_obs != nullptr);
    const int n = cfg->dev.N;
    const bool ten_by_ten = n >= 100 && n <= 128;
    // boards up to 10x10 with one observation issue the copy after the outcome (shipped-library sweeps, profiles/
    // r3o_shipped_tuning_sweep.txt, r3y_small_boards_tuning.txt: 8x8 +2.1 %, 6x6 +3.5 %, 5x5 +3.8 % over a late issue); both
    // observations and the 15x15 board issue late (15x15: 79.8 M late, 76.8 M after the outcome)
    const uint32_t ops = step_all_ops(out);
    const int issue = cfg->tune_issue >= 0 ? cfg->tune_issue
                    : compressed_warps_for(cfg, out, ops) ? 0
                    : (cfg->obs_elem_bytes == 2 && (ops & (OP_PO | OP_FO))) ? shape16(cfg->dev, ops).issue
                    : (n <= 128 && one_obs) ? 1 : 0;
    a.flags = (flags & 0xffffu) | (uint32_t(issue) << 20);
    if (issue == 0 && !ten_by_ten) a.flags |= SX_TUNE_COMMIT_GAP;  // late issue, not the 10x10 board
    a.out = out;
    a.ops = ops;
    a.setups = setups_d; a.n_setups = n_setups;
    a.key = make_key(seed);
    a.stats = reinterpret_cast<long long *>(stats_d);
    return launch_fused(cfg, a, static_cast<cudaStream_t>(stream));
}

extern "C" int sx_sample_valid(const uint8_t *mask_d, int64_t num_envs, int32_t mask_len, int64_t env_base, uint64_t seed,
                               uint32_t step, int32_t *actions_d, void *stream)
{
    if (!mask_d || !actions_d) return fail("sx_sample_valid: null argument");
    if (num_envs <= 0) return 0;
    const int wpb = 8;
    sx_sample_kernel<<<unsigned((num_envs + wpb - 1) / wpb), wpb * 32, 0, static_cast<cudaStream_t>(stream)>>>(
        mask_d, num_envs, mask_len, env_base, make_key(seed), step, actions_d);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail("sx_sample_kernel", e);
}

extern "C" int sx_heuristic_rewards(const sx_config *cfg, sx_state st, int64_t num_envs, const int32_t *actions_d,
                                    int32_t action_format, const float *reward_matrix_d, float *rewards_d, void *stream)
{
    if (int rc = check_state(cfg, st, "sx_heuristic_rewards")) return rc;
    if (!actions_d || !reward_matrix_d || !rewards_d) return fail("sx_heuristic_rewards: null argument");
    if (action_format != SX_ACTION_SPATIAL && action_format != SX_ACTION_1D) return fail("sx_heuristic_rewards: unknown action format");
    if (num_envs <= 0) return 0;
    const int threads = 256;
    sx_heuristic_kernel<<<unsigned((num_envs + threads - 1) / threads), threads, 0, static_cast<cudaStream_t>(stream)>>>(
        cfg->dev, st.board, st.aux, num_envs, actions_d, action_format, reward_matrix_d, rewards_d);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : cuda_fail("sx_heuristic_kernel", e);
}

extern "C" int sx_step_all_launch_info(const sx_config *cfg, uint32_t obs_mask, sx_launch_info *out)
{
    if (!cfg || !out) return fail("sx_step_all_launch_info: null argument");
    uint32_t ops = OP_STEP | OP_WRITE_STATE | OP_NEED_MOVES;
    if (obs_mask & 1) ops |= OP_PO;
    if (obs_mask & 2) ops |= OP_FO;
    if (obs_mask & 4) ops |= OP_MASK;
    LaunchPlan plan;
    KernelArgs probe;
    std::memset(&probe, 0, sizeof(probe));
    probe.ops = ops;
    probe.num_envs = 1LL << 40;
    out->thread_per_game = 0;
    if (toy_eligible(cfg, probe, mode_for(cfg, probe))) {  // the toy boards step through sx_toy_kernel
        ToyPlan tp;
        if (int rc = plan_toy(cfg, ops, &tp)) return rc;
        cudaFuncAttributes attr;
        cudaError_t e = cudaFuncGetAttributes(&attr, toy_for_mode(mode_for(cfg, probe), cfg->obs_elem_bytes));
        if (e != cudaSuccess) return cuda_fail("cudaFuncGetAttributes", e);
        out->warps_per_block = tp.warps; out->blocks_per_sm = 1; out->smem_bytes_per_block = tp.smem;
        out->num_sms = tp.num_sms; out->grid_blocks = tp.grid_max; out->regs_per_thread = attr.numRegs;
        out->background_bytes = tp.tile_bytes;
        out->thread_per_game = 1;
        return 0;
    }
    const int cw = (obs_mask & 8) ? compressed_shape_warps(cfg, ops) : 0;
    if (int rc = plan_launch(cfg, ops, mode_for(cfg, probe), 1LL << 40, &plan, cw)) return rc;
    out->warps_per_block = plan.warps_per_block; out->blocks_per_sm = plan.blocks_per_sm;
    out->smem_bytes_per_block = plan.smem_per_block; out->num_sms = plan.num_sms; out->grid_blocks = plan.grid;
    out->regs_per_thread = plan.regs;
    out->background_bytes = plan.tile_bytes;
    return 0;
}

// ---- host-buffer convenience object ------------------------------------------------------------------
struct sx_host_env {
    const sx_config *cfg;
    int64_t num_envs, env_base;
    uint32_t obs_mask, flags;
    uint64_t seed;
    int n_chunks;
    sx_state st;
    sx_outputs dev;        // device outputs, full batch
    int32_t *actions_d;
    uint8_t *setups_d;
    int32_t n_setups;
    int64_t *stats_d;
    std::vector<cudaStream_t> streams;
};

// every device buffer of the object comes from sx_device_alloc: the observation and mask planes compressible where the
// device grants it (they are written every step and are almost constant), the rest plain.  Below one 2 MB granule of
// compressible memory, compression would round up more than it saves (StrategoEngine applies the same bound).
template <typename T>
static cudaError_t dev_alloc(T **p, size_t count, uint32_t flags = 0)
{
    int device = 0;
    cudaError_t e = cudaGetDevice(&device);
    if (e != cudaSuccess) return e;
    void *q = nullptr;
    if (count * sizeof(T) < (size_t(2) << 20)) flags &= ~uint32_t(SX_ALLOC_COMPRESSIBLE);
    if (sx_device_alloc(device, count * sizeof(T), flags, &q, nullptr)) return cudaErrorMemoryAllocation;
    *p = static_cast<T *>(q);
    return cudaSuccess;
}

extern "C" void sx_host_env_destroy(sx_host_env *env)
{
    if (!env) return;
    for (cudaStream_t s : env->streams) cudaStreamDestroy(s);
    for (void *p : {static_cast<void *>(env->st.board), static_cast<void *>(env->st.aux), static_cast<void *>(env->st.captured),
                    static_cast<void *>(env->dev.partial_obs), static_cast<void *>(env->dev.full_obs),
                    static_cast<void *>(env->dev.valid_mask), static_cast<void *>(env->dev.reward),
                    static_cast<void *>(env->dev.done), static_cast<void *>(env->dev.winner),
                    static_cast<void *>(env->dev.ending_invalid), static_cast<void *>(env->dev.illegal),
                    static_cast<void *>(env->dev.player), static_cast<void *>(env->dev.next_action),
                    static_cast<void *>(env->actions_d), static_cast<void *>(env->setups_d), static_cast<void *>(env->stats_d)})
        sx_device_free(p);
    delete env;
}

extern "C" int sx_host_env_create(const sx_config *cfg, int64_t num_envs, int64_t env_base, uint32_t obs_mask, uint32_t flags,
                                  const uint8_t *setups_host, int32_t n_setups, uint64_t seed, int32_t n_chunks,
                                  sx_host_env **out)
{
    if (!cfg || !out || num_envs < 1) return fail("sx_host_env_create: bad argument");
    if (!(flags & SX_RESET_RANDOM_SHUFFLE) && (!setups_host || n_setups < 1))
        return fail("sx_host_env_create: a setup table or SX_RESET_RANDOM_SHUFFLE is required");
    sx_host_env *h = new (std::nothrow) sx_host_env();
    if (!h) return fail("out of memory");
    h->cfg = cfg; h->num_envs = num_envs; h->env_base = env_base; h->obs_mask = obs_mask; h->flags = flags; h->seed = seed;
    h->n_chunks = int(std::max<int64_t>(1, std::min<int64_t>(n_chunks, num_envs)));
    h->n_setups = n_setups;
    const DevConfig &d = cfg->dev;
    const size_t B = size_t(num_envs);
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    ok(dev_alloc(&h->st.board, B * d.board_stride));
    ok(dev_alloc(&h->st.aux, B * 8));
    ok(dev_alloc(&h->st.captured, B * d.cap_stride));
    const size_t eb = size_t(cfg->obs_elem_bytes);
    if (obs_mask & 1) ok(dev_alloc(reinterpret_cast<uint8_t **>(&h->dev.partial_obs), B * d.po_floats * eb, SX_ALLOC_COMPRESSIBLE));
    if (obs_mask & 2) ok(dev_alloc(reinterpret_cast<uint8_t **>(&h->dev.full_obs), B * d.fo_floats * eb, SX_ALLOC_COMPRESSIBLE));
    if (obs_mask & 4) ok(dev_alloc(&h->dev.valid_mask, B * d.mask_bytes, SX_ALLOC_COMPRESSIBLE));
    ok(dev_alloc(&h->dev.reward, B)); ok(dev_alloc(&h->dev.done, B)); ok(dev_alloc(&h->dev.winner, B));
    ok(dev_alloc(&h->dev.ending_invalid, B)); ok(dev_alloc(&h->dev.illegal, B)); ok(dev_alloc(&h->dev.player, B));
    ok(dev_alloc(&h->dev.next_action, B));
    ok(dev_alloc(&h->actions_d, B));
    ok(dev_alloc(&h->stats_d, 8));
    if (setups_host && n_setups > 0) {
        ok(dev_alloc(&h->setups_d, size_t(n_setups) * d.setup_len));
        if (e == cudaSuccess) ok(cudaMemcpy(h->setups_d, setups_host, size_t(n_setups) * d.setup_len, cudaMemcpyHostToDevice));
    }
    if (e == cudaSuccess) ok(cudaMemset(h->st.aux, 0, B * 8 * sizeof(int16_t)));
    if (e == cudaSuccess) ok(cudaMemset(h->stats_d, 0, 8 * sizeof(int64_t)));
    const int n_streams = std::min(h->n_chunks, 4);
    for (int i = 0; i < n_streams && e == cudaSuccess; ++i) {
        cudaStream_t s;
        ok(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
        if (e == cudaSuccess) h->streams.push_back(s);
    }
    if (e != cudaSuccess) {
        sx_host_env_destroy(h);
        return cuda_fail("sx_host_env_create", e);
    }
    *out = h;
    return 0;
}

static sx_state offset_state(const sx_host_env *h, int64_t lo)
{
    const DevConfig &d = h->cfg->dev;
    return sx_state{h->st.board + lo * d.board_stride, h->st.aux + lo * 8, h->st.captured + lo * d.cap_stride};
}

template <typename T>
static cudaError_t d2h(T *host, const T *dev, size_t count, cudaStream_t s)
{
    if (!host || !dev) return cudaSuccess;
    return cudaMemcpyAsync(host, dev, count * sizeof(T), cudaMemcpyDeviceToHost, s);
}

static int copy_outputs(const sx_host_env *h, const sx_outputs &host, int64_t lo, int64_t n, cudaStream_t s)
{
    const DevConfig &d = h->cfg->dev;
    const size_t eb = size_t(h->cfg->obs_elem_bytes);
    const sx_outputs dv = offset_outputs(h->cfg, h->dev, lo), hv = offset_outputs(h->cfg, host, lo);
    cudaError_t e = cudaSuccess;
    auto ok = [&](cudaError_t r) { if (e == cudaSuccess) e = r; };
    auto bytes = [](float *p) { return reinterpret_cast<uint8_t *>(p); };
    ok(d2h(bytes(hv.partial_obs), bytes(dv.partial_obs), size_t(n) * d.po_floats * eb, s));
    ok(d2h(bytes(hv.full_obs), bytes(dv.full_obs), size_t(n) * d.fo_floats * eb, s));
    ok(d2h(hv.valid_mask, dv.valid_mask, size_t(n) * d.mask_bytes, s));
    ok(d2h(hv.reward, dv.reward, size_t(n), s));
    ok(d2h(hv.done, dv.done, size_t(n), s));
    ok(d2h(hv.winner, dv.winner, size_t(n), s));
    ok(d2h(hv.ending_invalid, dv.ending_invalid, size_t(n), s));
    ok(d2h(hv.illegal, dv.illegal, size_t(n), s));
    ok(d2h(hv.player, dv.player, size_t(n), s));
    ok(d2h(hv.next_action, dv.next_action, size_t(n), s));
    return e == cudaSuccess ? 0 : cuda_fail("sx_host_env D2H", e);
}

extern "C" int sx_host_env_state(sx_host_env *env, sx_state *state_out, sx_outputs *device_outputs_out)
{
    if (!env || !state_out) return fail("sx_host_env_state: null argument");
    *state_out = env->st;
    if (device_outputs_out) *device_outputs_out = env->dev;
    return 0;
}

extern "C" int sx_host_env_sync(sx_host_env *env)
{
    if (!env) return fail("sx_host_env_sync: null env");
    for (cudaStream_t s : env->streams) {
        cudaError_t e = cudaStreamSynchronize(s);
        if (e != cudaSuccess) return cuda_fail("cudaStreamSynchronize", e);
    }
    return 0;
}

extern "C" int sx_host_env_reset(sx_host_env *h, sx_outputs host_out)
{
    if (!h) return fail("sx_host_env_reset: null env");
    for (int c = 0; c < h->n_chunks; ++c) {
        const int64_t lo = h->num_envs * c / h->n_chunks, hi = h->num_envs * (c + 1) / h->n_chunks;
        cudaStream_t s = h->streams[c % h->streams.size()];
        if (int rc = sx_reset(h->cfg, offset_state(h, lo), hi - lo, h->env_base + lo, nullptr, h->setups_d, h->n_setups, nullptr,
                              h->seed, h->flags & (SX_RESET_RANDOM_SHUFFLE | SX_SAME_SETUP | SX_REPEAT_OTHER_SIDE), s))
            return rc;
        sx_outputs o = offset_outputs(h->cfg, h->dev, lo);
        KernelArgs a;
        base_args(a, offset_state(h, lo), hi - lo, h->env_base + lo);
        a.out = o;
        a.flags = h->flags & SX_SAMPLE_NEXT;
        a.key = make_key(h->seed);
        a.ops = (o.valid_mask ? OP_MASK : 0) | (o.partial_obs ? OP_PO : 0) | (o.full_obs ? OP_FO : 0) | OP_NEED_MOVES;
        if (int rc = launch_fused(h->cfg, a, s)) return rc;
        if (int rc = copy_outputs(h, host_out, lo, hi - lo, s)) return rc;
    }
    return sx_host_env_sync(h);
}

static int host_env_step_impl(sx_host_env *h, const int32_t *actions_host, const int32_t *actions_dev_src,
                              const sx_outputs *host_out, int action_format = SX_ACTION_SPATIAL, int64_t flags = -1)
{
    const uint32_t step_flags = flags < 0 ? h->flags : uint32_t(flags);
    for (int c = 0; c < h->n_chunks; ++c) {
        const int64_t lo = h->num_envs * c / h->n_chunks, hi = h->num_envs * (c + 1) / h->n_chunks;
        cudaStream_t s = h->streams[c % h->streams.size()];
        const int32_t *acts = actions_dev_src ? actions_dev_src + lo : h->actions_d + lo;
        if (actions_host) {
            cudaError_t e = cudaMemcpyAsync(h->actions_d + lo, actions_host + lo, size_t(hi - lo) * sizeof(int32_t),
                                            cudaMemcpyHostToDevice, s);
            if (e != cudaSuccess) return cuda_fail("sx_host_env H2D", e);
        }
        if (int rc = sx_step_all(h->cfg, offset_state(h, lo), hi - lo, h->env_base + lo, acts, action_format, step_flags,
                                 h->setups_d, h->n_setups, h->seed, offset_outputs(h->cfg, h->dev, lo), h->stats_d, s))
            return rc;
        if (host_out)
            if (int rc = copy_outputs(h, *host_out, lo, hi - lo, s)) return rc;
    }
    return 0;
}

extern "C" int sx_host_env_step(sx_host_env *h, const int32_t *actions_host, sx_outputs host_out)
{
    if (!h || !actions_host) return fail("sx_host_env_step: null argument");
    if (int rc = host_env_step_impl(h, actions_host, nullptr, &host_out)) return rc;
    return sx_host_env_sync(h);
}

extern "C" int sx_host_env_step_ex(sx_host_env *h, const int32_t *actions_host, int32_t action_format, uint32_t flags,
                                   sx_outputs host_out)
{
    if (!h || !actions_host) return fail("sx_host_env_step_ex: null argument");
    if (action_format != SX_ACTION_SPATIAL && action_format != SX_ACTION_1D) return fail("sx_host_env_step_ex: unknown action format");
    if (int rc = host_env_step_impl(h, actions_host, nullptr, &host_out, action_format, int64_t(flags))) return rc;
    return sx_host_env_sync(h);
}

extern "C" int sx_host_env_step_device(sx_host_env *h, int32_t use_sampled_actions)
{
    if (!h) return fail("sx_host_env_step_device: null env");
    if (use_sampled_actions) {
        // the sampled actions of the previous step become this step's input (device to device, same stream order)
        for (int c = 0; c < h->n_chunks; ++c) {
            const int64_t lo = h->num_envs * c / h->n_chunks, hi = h->num_envs * (c + 1) / h->n_chunks;
            cudaStream_t s = h->streams[c % h->streams.size()];
            cudaError_t e = cudaMemcpyAsync(h->actions_d + lo, h->dev.next_action + lo, size_t(hi - lo) * sizeof(int32_t),
                                            cudaMemcpyDeviceToDevice, s);
            if (e != cudaSuccess) return cuda_fail("sx_host_env D2D", e);
        }
    }
    return host_env_step_impl(h, nullptr, nullptr, nullptr);
}
