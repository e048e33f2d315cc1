// sx_device.cuh -- device-side game logic of the B200 Stratego engine (one warp per game).
//
// Everything here is warp-synchronous: the 32 lanes of a warp cooperate on ONE game whose compact
// state is staged in that warp's slice of shared memory.  Scalar rule logic (action decode, combat)
// is computed redundantly by all lanes (warp-uniform control flow, one issue slot per op); board
// scans are spread over lanes, K = ceil(cells / 32) consecutive cells per lane.
//
// Reference being restated: stratego_env/game/stratego_procedural_impl.py ("impl") and
// stratego_env/stratego_multiagent_env.py ("maenv") of JBLanier/stratego_env.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/stratego_b200.h"

// The per-lane cell loops (k < K) of the hot functions stay rolled (`#pragma unroll 1`): that keeps the fused loop small
// enough for the instruction cache; unrolling them cost 9 % on Barrage / Standard (profiles/r2n_register_budget_sweep.txt).

namespace sx {

// ---- piece codes (impl:145-163) -----------------------------------------------------------------
constexpr int SP_SPY = 1, SP_SCOUT = 2, SP_MINER = 3, SP_MARSHAL = 10, SP_FLAG = 11, SP_BOMB = 12, SP_UNKNOWN = 13;

// ---- packed board cell: one byte per square ------------------------------------------------------
// Sufficient because on every reachable state the partially observable rank is either UNKNOWN or the
// true rank (impl:955-995), so the reference's six per-cell layers (true rank x2, PO rank x2, still
// x2) plus the obstacle layer collapse to rank/owner/revealed/still/obstacle.
constexpr uint32_t CELL_RANK = 0x0F, CELL_OWNER = 0x10, CELL_REVEALED = 0x20, CELL_STILL = 0x40, CELL_OBST = 0x80;

constexpr int NO_CELL = 255;
constexpr uint32_t FULL = 0xffffffffu;

// ---- per-variant constants, passed by value as a kernel parameter ---------------------------------
struct DevConfig {
    int R, C, N, A, mpa, action_size;
    int board_stride, cap_stride;  // bytes / uint16 entries per env
    int max_turns, usable_rows, setup_len, n_pieces, p2_rot180;
    uint32_t magic_C, magic_A, magic_mpa;  // floor(2^32 / d) + 1: x / d == __umulhi(x, magic) for x * d < 2^32
    int po_floats, fo_floats, mask_bytes;
    float cap_lut[12 * 9];
    float recent_lut[5];
    float unit_lut[2];
    // deprecated 'original' channel mode (maenv:370-375): one channel per state layer carrying the normalised raw value
    int original_channels, po_ch, fo_ch;  // po_ch / fo_ch: channels of the two observations (67 / 79 or 32 / 33)
    float rank_lut[14];     // normalised true-rank value 0..12 (maenv:88-89)
    float po_rank_lut[14];  // normalised partially observable rank 0..13 (maenv:91-92)
    uint8_t obstacles[256];
    uint8_t piece_seq[128];  // pieces in placement order (piece code ascending, util:24-28)
};

// Two small values indexed by player (0 / 1).  A plain `int x[2]` indexed with a run-time player index makes the
// compiler put the whole Aux object into local memory (85 LDL / STL instructions in the thread-per-game kernel, ~100 in
// the warp-level ones); this keeps both values in registers and turns the index into a select.
struct PerPlayer {
    int v0, v1;
    struct Ref {
        int &v0, &v1;
        int i;
        __device__ __forceinline__ operator int() const { return i ? v1 : v0; }
        __device__ __forceinline__ int operator=(int x) { if (i) v1 = x; else v0 = x; return x; }
        __device__ __forceinline__ int operator=(const Ref &o) { return *this = int(o); }
    };
    __device__ __forceinline__ Ref operator[](int i) { return Ref{v0, v1, i}; }
    __device__ __forceinline__ int operator[](int i) const { return i ? v1 : v0; }
};

// ---- scalar part of a game's state (aux tensor, 8 x int16) ----------------------------------------
struct Aux {
    int turn, max_turns;
    int over, invalid, winner;  // winner in {-1, 0, +1}
    int to_move;                // 0 = player +1, 1 = player -1
    PerPlayer rfrom, rto, rcode;  // recent-move squares per player (NO_CELL = none); rcode = -code of `to` (1..3)
    int ncap;
    int overflow;               // sticky: a capture did not fit the capture list -> the compact state lost information
    uint32_t episode;
};

__device__ __forceinline__ void aux_unpack(const uint32_t w[4], Aux &a)
{
    a.turn = w[0] & 0xffff;
    a.max_turns = w[0] >> 16;
    const uint32_t flags = w[1] & 0xff;
    a.over = flags & 1;
    a.invalid = (flags >> 1) & 1;
    a.winner = int((flags >> 2) & 3) - 1;
    a.to_move = (flags >> 4) & 1;
    a.overflow = (flags >> 5) & 1;
    a.ncap = (w[1] >> 8) & 0xff;
    a.rfrom[0] = (w[1] >> 16) & 0xff;
    a.rto[0] = (w[1] >> 24) & 0xff;
    a.rfrom[1] = w[2] & 0xff;
    a.rto[1] = (w[2] >> 8) & 0xff;
    a.rcode[0] = (w[2] >> 16) & 0xff;
    a.rcode[1] = (w[2] >> 24) & 0xff;
    a.episode = w[3];
}

__device__ __forceinline__ void aux_pack(const Aux &a, uint32_t w[4])
{
    w[0] = uint32_t(a.turn & 0xffff) | (uint32_t(a.max_turns & 0xffff) << 16);
    const uint32_t flags = uint32_t(a.over) | (uint32_t(a.invalid) << 1) | (uint32_t(a.winner + 1) << 2) |
                           (uint32_t(a.to_move) << 4) | (uint32_t(a.overflow) << 5);
    w[1] = flags | (uint32_t(a.ncap) << 8) | (uint32_t(a.rfrom[0]) << 16) | (uint32_t(a.rto[0]) << 24);
    w[2] = uint32_t(a.rfrom[1]) | (uint32_t(a.rto[1]) << 8) | (uint32_t(a.rcode[0]) << 16) |
           (uint32_t(a.rcode[1]) << 24);
    w[3] = a.episode;
}

// capture entry: cell | owner<<8 | (type-1)<<9 | (count-1)<<13
__device__ __forceinline__ uint32_t cap_key(int cell, int owner, int type) { return uint32_t(cell) | (uint32_t(owner) << 8) | (uint32_t(type - 1) << 9); }

// ---- Philox4x32-10 (counter-based; results depend only on key/counter, not on placement) -----------
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u;
        k.y += 0xBB67AE85u;
    }
    return c;
}

enum : uint32_t { RNG_RESET = 0x52535430u, RNG_SAMPLE = 0x53414d50u, RNG_SHUFFLE = 0x53484600u, RNG_HIDDEN = 0x48494444u,
                  RNG_KEYS = 0x4b455953u, RNG_SEARCH = 0x54524545u };

// ---- this warp's slice of shared memory -----------------------------------------------------------
struct WarpMem {
    uint8_t *board;    // [board_stride]
    uint16_t *cap;     // [cap_stride]
    uint32_t *lines;   // [64] occupancy bit-lines: any[0..15 rows | 16..31 cols], enemy[32 + same]
    uint2 *moves;      // [N] per-cell 64-bit set of playable spatial channels: the move list the outputs are built from
    uint8_t *scratch;  // [>= 2 * setup_len] shuffle workspace
};

__host__ __device__ inline int round16(int v) { return (v + 15) & ~15; }

// shared-memory slice of one warp; host and device must agree on this layout
__host__ __device__ inline int carve_warp(const DevConfig &cfg, uint8_t *base, WarpMem *m)
{
    int off = 0;
    if (m) m->board = base + off;
    off += cfg.board_stride;
    if (m) m->cap = reinterpret_cast<uint16_t *>(base + off);
    off += round16(cfg.cap_stride * 2);
    if (m) m->lines = reinterpret_cast<uint32_t *>(base + off);
    off += 256;
    if (m) m->moves = reinterpret_cast<uint2 *>(base + off);
    off += round16(cfg.N * 8);
    if (m) m->scratch = base + off;
    off += round16(2 * cfg.setup_len);
    return off;
}


// The block's read-only background images: what a game's outputs look like before the state-dependent
// entries are added ("empty board" observation after normalisation; all-zero mask).
struct Tile {
    float *po;      // [N*67] partial observation
    float *fo;      // [N*79] full observation
    uint8_t *mask;  // [mask_bytes + 16] zeros; copies start at mask + (global address & 15)
};

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// ---- games per warp ------------------------------------------------------------------------------------
// A 10x10 board uses all 32 lanes of a warp; the toy variants (3x4 ... 5x5) would leave most lanes idle and
// replicate the scalar rule logic 32 times for 12-25 cells.  For those, G = 2 or 4 games share a warp: each
// game owns a contiguous group of L = 32 / G lanes, every warp-level primitive below is restricted to the
// group's lane mask, and the (identical) instruction stream advances G games at once.
template <int G>
struct Grp {
    static constexpr int GAMES = G;
    static constexpr int L = 32 / G;  // lanes per game
    static constexpr int H = L / 2;   // lanes building row lines; the other half builds column lines
    static __device__ __forceinline__ int lane() { return threadIdx.x & (L - 1); }
    static __device__ __forceinline__ int index() { return (threadIdx.x & 31) / L; }
    static __device__ __forceinline__ uint32_t mask()
    {
        return G == 1 ? FULL : ((G == 2 ? 0xffffu : 0xffu) << (index() * L));
    }
    static __device__ __forceinline__ void sync() { __syncwarp(mask()); }
    static __device__ __forceinline__ bool any(int pred) { return __any_sync(mask(), pred) != 0; }
    static __device__ __forceinline__ uint32_t ballot(int pred) { return __ballot_sync(mask(), pred) >> (index() * L); }
    static __device__ __forceinline__ int shfl(int v, int src) { return __shfl_sync(mask(), v, src, L); }
    static __device__ __forceinline__ int shfl_up(int v, int delta) { return __shfl_up_sync(mask(), v, delta, L); }
};
__device__ __forceinline__ int fast_div(int x, uint32_t magic) { return int(__umulhi(uint32_t(x), magic)); }

// flat cell index in `me`'s frame <-> absolute frame: a 180-degree rotation is index reversal
__device__ __forceinline__ int view(int cell, int flip, int N) { return flip ? N - 1 - cell : cell; }

// ---- TMA bulk copy shared -> global (SASS: UBLKCP), tracked by the issuing thread's bulk group -----
// Stores and copies carry no L2 cache hint: state evict_last + outputs evict_first measured < 2 % on Barrage and -10 % on
// Standard, the reverse policy -2 to -5 % (DESIGN.md §3.1).
__device__ __forceinline__ void bulk_store(void *gdst, const void *ssrc, uint32_t bytes)
{
    const uint32_t saddr = static_cast<uint32_t>(__cvta_generic_to_shared(ssrc));
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(saddr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_but_one() { asm volatile("cp.async.bulk.wait_group 1;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Emits `bytes` from shared memory to global memory.  When src and dst are congruent mod 16 the
// 16-byte aligned body goes out as one TMA bulk copy issued by lane 0 (caller commits/waits) and the
// <16-byte head and tail as plain word stores; otherwise (odd-sized variants such as 5x5 and 15x15,
// whose per-env byte counts are not multiples of 16) the tile is copied with plain stores.
template <class GT>
static __device__ __noinline__ void emit_tile(uint8_t *gdst, const uint8_t *ssrc, int bytes)
{
    const int lane = GT::lane();
    const uintptr_t g = reinterpret_cast<uintptr_t>(gdst);
    const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(ssrc));
    if (((g | s | uint32_t(bytes)) & 3) != 0) {
        for (int i = lane; i < bytes; i += GT::L) gdst[i] = ssrc[i];
        return;
    }
    if (((g ^ s) & 15) != 0) {
        for (int i = lane; i < (bytes >> 2); i += GT::L)
            reinterpret_cast<uint32_t *>(gdst)[i] = reinterpret_cast<const uint32_t *>(ssrc)[i];
        return;
    }
    int head = int((16 - (g & 15)) & 15);
    if (head > bytes) head = bytes;
    const int body = (bytes - head) & ~15;
    const int tail = bytes - head - body;
    if (lane < (head >> 2)) reinterpret_cast<uint32_t *>(gdst)[lane] = reinterpret_cast<const uint32_t *>(ssrc)[lane];
    if (lane >= 4 && lane - 4 < (tail >> 2)) {
        const int off = head + body + ((lane - 4) << 2);
        *reinterpret_cast<uint32_t *>(gdst + off) = *reinterpret_cast<const uint32_t *>(ssrc + off);
    }
    if (body > 0 && lane == 0) bulk_store(gdst + head, ssrc + head, uint32_t(body));
}

// emit_tile for 16-bit observations: src, dst and bytes are even, and the callers pick a source congruent to the
// destination mod 16 (align_cells16), so the head and tail (at most 7 half-words each; a lane group has >= 8 lanes)
// go out as one half-word store per lane and the body as one TMA bulk copy.  A destination no image row can match (a
// caller's buffer that starts inside a 64-byte cell of the 32-channel mode) is copied with half-word stores.
template <class GT>
static __device__ __noinline__ void emit_tile16(uint8_t *gdst, const uint8_t *ssrc, int bytes)
{
    const int lane = GT::lane();
    const uintptr_t g = reinterpret_cast<uintptr_t>(gdst);
    const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(ssrc));
    uint16_t *gd = reinterpret_cast<uint16_t *>(gdst);
    const uint16_t *sd = reinterpret_cast<const uint16_t *>(ssrc);
    if (((g ^ s) & 15) != 0) {
        for (int i = lane; i < (bytes >> 1); i += GT::L) gd[i] = sd[i];
        return;
    }
    int head = int((16 - (g & 15)) & 15);
    if (head > bytes) head = bytes;
    const int body = (bytes - head) & ~15;
    const int tail_at = (head + body) >> 1;
    if (lane < (head >> 1)) gd[lane] = sd[lane];
    if (lane < ((bytes - head - body) >> 1)) gd[tail_at + lane] = sd[tail_at + lane];
    if (body > 0 && lane == 0) bulk_store(gdst + head, ssrc + head, uint32_t(body));
}

// ---- occupancy bit-lines in `me`'s frame ------------------------------------------------------------
// the first half of a game's lanes build one row each (bit c), the second half one column each (bit r);
// "any" marks pieces and lakes, "enemy" marks the opponent's pieces.  Replaces the per-square ray walk of
// impl:426-490.  Layout of m.lines: any[0..H) rows, any[H..L) columns, enemy at L + the same.
template <class GT>
__device__ __forceinline__ void build_lines(const DevConfig &cfg, const WarpMem &m, int me, int flip)
{
    const int lane = GT::lane();
    const bool is_row = lane < GT::H;
    const int idx = is_row ? lane : lane - GT::H;
    const int count = is_row ? cfg.C : cfg.R;
    const int stride = is_row ? 1 : cfg.C;
    const int base = is_row ? idx * cfg.C : idx;
    const bool live = idx < (is_row ? cfg.R : cfg.C);
    uint32_t any = 0, enemy = 0;
    if (live) {
        for (int j = 0; j < count; ++j) {
            const uint32_t b = m.board[view(base + j * stride, flip, cfg.N)];
            any |= uint32_t(b != 0) << j;
            enemy |= uint32_t((b & CELL_RANK) != 0 && int((b >> 4) & 1) != me) << j;
        }
    }
    m.lines[lane] = any;
    m.lines[GT::L + lane] = enemy;
    GT::sync();
}

// distance a sliding piece can travel from bit `pos` towards higher / lower bits of a line; the last
// square counts when it holds an enemy piece (impl:434-437, 454-456)
__device__ __forceinline__ int ray_up(uint32_t any, uint32_t enemy, int pos, int len)
{
    const uint32_t x = any >> (pos + 1);
    if (x == 0) return len - 1 - pos;
    const int d = __ffs(x);
    return (d - 1) + int((enemy >> (pos + d)) & 1);
}
__device__ __forceinline__ int ray_down(uint32_t any, uint32_t enemy, int pos)
{
    const uint32_t x = any & ((1u << pos) - 1u);
    if (x == 0) return pos;
    const int top = 31 - __clz(x);
    return (pos - top - 1) + int((enemy >> top) & 1);
}

// The single move the two-square rule can forbid for the player to move (impl:439-445, 501-505):
// from the square coded -3 back onto the square coded +1, if that square is empty.
struct Blocked {
    int cell, dir, dist;  // in `me`'s frame; cell < 0 = nothing blocked
};

__device__ __forceinline__ Blocked blocked_move(const DevConfig &cfg, const WarpMem &m, const Aux &a, int me, int flip,
                                                bool allow_osc)
{
    Blocked b{-1, 0, 0};
    if (allow_osc || a.rcode[me] != 3 || a.rto[me] == NO_CELL || a.rfrom[me] == NO_CELL) return b;
    if ((m.board[a.rfrom[me]] & CELL_RANK) != 0) return b;  // an enemy stepped onto it: attacking is allowed
    const int s = view(a.rto[me], flip, cfg.N), e = view(a.rfrom[me], flip, cfg.N);
    const int sr = fast_div(s, cfg.magic_C), sc = s - sr * cfg.C, er = fast_div(e, cfg.magic_C), ec = e - er * cfg.C;
    if (sr != er && sc != ec) return b;
    if (s == e) return b;
    b.cell = s;
    if (sc == ec) { b.dir = er > sr ? 0 : 1; b.dist = er > sr ? er - sr : sr - er; }
    else { b.dir = ec > sc ? 2 : 3; b.dist = ec > sc ? ec - sc : sc - ec; }
    return b;
}

// ---- valid-move generation (impl:400-517 / impl:522-642) -------------------------------------------
// Move generation produces, per cell, a 64-bit set over the spatial channels (bit ch = "the piece on this
// cell may play channel ch", channel layout impl:292-311) in m.moves, with the one move the two-square rule
// forbids already removed.  The spatial mask, the 1D mask and the uniform sampler are expansions of it.
__device__ __forceinline__ int dir_base(const DevConfig &cfg, int dir)  // first channel of a direction, impl:292-311
{
    return dir == 0 ? 0 : dir == 1 ? (cfg.R - 1) : dir == 2 ? 2 * (cfg.R - 1) : 2 * (cfg.R - 1) + (cfg.C - 1);
}

// Enumerates the moves of player index `me`, in `me`'s frame, into m.moves.  Returns (warp-uniform)
// whether any move exists.
template <int K, class GT, bool COMPACT = false>
__device__ __forceinline__ bool gen_moves(const DevConfig &cfg, const WarpMem &m, const Aux &a, int me, bool allow_osc)
{
    const int lane = GT::lane();
    if (a.over) {  // impl:414
#pragma unroll 1
        for (int k = 0; k < K; ++k) {
            const int p = lane * K + k;
            if (p < cfg.N) m.moves[p] = make_uint2(0, 0);
        }
        GT::sync();
        return false;
    }
    const int flip = me;  // player -1 sees the board rotated
    build_lines<GT>(cfg, m, me, flip);
    const Blocked blk = blocked_move(cfg, m, a, me, flip, allow_osc);
    const int b1 = cfg.R - 1, b2 = 2 * b1, b3 = b2 + cfg.C - 1;
    const int blocked_bit = blk.cell < 0 ? 0 : (blk.dir == 0 ? 0 : blk.dir == 1 ? b1 : blk.dir == 2 ? b2 : b3) + blk.dist - 1;
    // the moves of the piece on cell p (a piece of `me` that can move, impl:420), two-square rule applied
    auto piece_moves = [&](int p, int rank) {
        const int r = fast_div(p, cfg.magic_C), c = p - r * cfg.C;
        const uint32_t col_any = m.lines[GT::H + c], col_en = m.lines[GT::L + GT::H + c];
        const uint32_t row_any = m.lines[r], row_en = m.lines[GT::L + r];
        int n0 = ray_up(col_any, col_en, r, cfg.R), n1 = ray_down(col_any, col_en, r);
        int n2 = ray_up(row_any, row_en, c, cfg.C), n3 = ray_down(row_any, row_en, c);
        if (rank != SP_SCOUT) { n0 = min(n0, 1); n1 = min(n1, 1); n2 = min(n2, 1); n3 = min(n3, 1); }  // impl:492-499
        unsigned long long bits = (unsigned long long)((1u << n0) - 1u) | ((unsigned long long)((1u << n1) - 1u) << b1) |
                                  ((unsigned long long)((1u << n2) - 1u) << b2) | ((unsigned long long)((1u << n3) - 1u) << b3);
        if (p == blk.cell) bits &= ~(1ull << blocked_bit);  // impl:439-445, 501-505
        return bits;
    };
    int found = 0;
    if constexpr (COMPACT) {
        // Dense big boards (Standard: up to 33 movable pieces on 100 cells): a cell-major loop runs the ray arithmetic K
        // times because SOME lane has a mover each time.  Instead the lanes classify their cells (one ballot per k), mover
        // number t goes to lane t, and the ray arithmetic runs once per 32 movers.  Measured (profiles/r3g_*, r3j_*):
        // Standard 168.5 -> 175.8 M env-steps/s, the state-based sampler 0.194 -> 0.162 ms, the mask kernel 0.252 -> 0.206
        // ms; on a sparse board (Barrage, 8 pieces) the ballots cost what the loop did and the 170 extra hot instructions
        // raise the instruction-fetch stalls (185.8 -> 180.3 M), so the host picks per variant (sx_config::compact_movers).
        uint32_t movers[K];
        int total = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const int p = lane * K + k;
            bool mv = false;
            if (p < cfg.N) {
                const uint32_t b = m.board[view(p, flip, cfg.N)];
                const int rank = b & CELL_RANK;
                mv = rank != 0 && rank <= SP_MARSHAL && int((b >> 4) & 1) == me;
                m.moves[p] = make_uint2(0, 0);
            }
            movers[k] = GT::ballot(mv);
            total += __popc(movers[k]);
        }
        GT::sync();
        for (int t = lane; t < total; t += GT::L) {
            int r = t, k = 0;
#pragma unroll
            for (int j = 0; j + 1 < K; ++j) {  // which k-class mover t falls in, and its number inside the class
                const int c = __popc(movers[j]);
                if (k == j && r >= c) { r -= c; k = j + 1; }
            }
            uint32_t mk = movers[0];
#pragma unroll
            for (int j = 1; j < K; ++j) mk = k == j ? movers[j] : mk;
            const int p = int(__fns(mk, 0, r + 1)) * K + k;
            const unsigned long long bits = piece_moves(p, m.board[view(p, flip, cfg.N)] & CELL_RANK);
            found |= bits != 0;
            m.moves[p] = make_uint2(uint32_t(bits), uint32_t(bits >> 32));
        }
    } else {
#pragma unroll 1
        for (int k = 0; k < K; ++k) {
            const int p = lane * K + k;
            if (p < cfg.N) {
                unsigned long long bits = 0;
                const uint32_t b = m.board[view(p, flip, cfg.N)];
                const int rank = b & CELL_RANK;
                if (rank != 0 && rank <= SP_MARSHAL && int((b >> 4) & 1) == me) {  // impl:420
                    bits = piece_moves(p, rank);
                    found |= bits != 0;
                }
                m.moves[p] = make_uint2(uint32_t(bits), uint32_t(bits >> 32));
            }
        }
    }
    GT::sync();
    return GT::any(found);
}

// Expands m.moves into the spatial mask [cell][channel]: stores a 1 at every move on top of the zero
// background at `image` (global memory).
template <int K, class GT>
__device__ __forceinline__ void mark_spatial(const DevConfig &cfg, const WarpMem &m, uint8_t *image)
{
    const int lane = GT::lane();
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        const uint2 bits = p < cfg.N ? m.moves[p] : make_uint2(0, 0);
        if ((bits.x | bits.y) != 0) {
            uint8_t *cell = image + p * cfg.A;
#pragma unroll 1
            for (uint32_t w = bits.x; w != 0; w &= w - 1) *(cell + __ffs(w) - 1) = 1;
#pragma unroll 1
            for (uint32_t w = bits.y; w != 0; w &= w - 1) *(cell + 31 + __ffs(w)) = 1;
        }
    }
}

// Expands m.moves into a 1D mask row in global memory, absolute frame (impl:264-277); facade use only.
template <int K, class GT>
static __device__ __noinline__ void mark_1d_global(const DevConfig *cfgp, const uint2 *moves, int flip, uint8_t *row)
{
    const DevConfig &cfg = *cfgp;
    const int lane = GT::lane();
    const int b1 = cfg.R - 1, b2 = 2 * b1, b3 = b2 + cfg.C - 1;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p >= cfg.N) continue;
        const int r = fast_div(p, cfg.magic_C), c = p - r * cfg.C;
        const int s = view(p, flip, cfg.N);
        unsigned long long bits = (unsigned long long)moves[p].x | ((unsigned long long)moves[p].y << 32);
#pragma unroll 1
        for (; bits != 0; bits &= bits - 1) {
            const int ch = __ffsll((long long)bits) - 1;
            const int d = ch >= b3 ? 3 : ch >= b2 ? 2 : ch >= b1 ? 1 : 0;
            const int t = ch - (d == 0 ? 0 : d == 1 ? b1 : d == 2 ? b2 : b3) + 1;
            int er = r, ec = c;  // target in `me`'s frame
            if (d == 0) er += t; else if (d == 1) er -= t; else if (d == 2) ec += t; else ec -= t;
            if (flip) { er = cfg.R - 1 - er; ec = cfg.C - 1 - ec; }
            row[s * cfg.mpa + (d < 2 ? er : cfg.R + ec)] = 1;
        }
    }
}

// ---- action decode ----------------------------------------------------------------------------------
struct Move {
    int start, end;      // absolute cells
    int sr, sc, er, ec;  // their absolute rows / columns
    bool noop, bad;
};

// absolute 1D index (impl:352-383); the last index is the noop.  Anything outside [0, action_size) decodes in the
// reference (floor division) to a start square off the board, which impl:745-749 rejects.
__device__ __forceinline__ Move decode_1d(const DevConfig &cfg, int action)
{
    Move mv{0, 0, 0, 0, 0, 0, false, true};
    if (action == cfg.action_size - 1) { mv.noop = true; mv.bad = false; return mv; }
    if (action < 0 || action >= cfg.action_size) return mv;
    const int cell = fast_div(action, cfg.magic_mpa), off = action - cell * cfg.mpa;
    const int r = fast_div(cell, cfg.magic_C), c = cell - r * cfg.C;
    const int er = off >= cfg.R ? r : off, ec = off >= cfg.R ? off - cfg.R : c;
    mv.sr = r; mv.sc = c; mv.er = er; mv.ec = ec;
    mv.start = cell;
    mv.end = er * cfg.C + ec;
    mv.bad = false;
    return mv;
}

// Python's // and % (numba int64 floor semantics) for a possibly negative numerator and d > 0
__device__ __forceinline__ int floor_div(int x, int d) { const int q = x / d; return (x % d != 0 && x < 0) ? q - 1 : q; }
__device__ __forceinline__ int floor_mod(int x, int d) { const int m = x % d; return m < 0 ? m + d : m; }

// A spatial action whose target square is off the board, or that uses the noop channel.  The reference does NOT
// reject these: impl:316-335 produces the unchecked target, impl:264-277 folds it into a 1D index that ALIASES another
// move (or the 1D noop, or an index outside the action space), impl:700-720 rotates that index for player -1 with
// floor division, and _get_next_state plays whatever it decodes to (impl:803-831).  Reproduced step by step; cold.
static __device__ __noinline__ int alias_spatial_1d(const DevConfig *cfgp, int cell, int r, int er, int ec, int flip)
{
    const DevConfig &cfg = *cfgp;
    int idx = cell * cfg.mpa + (er != r ? er : cfg.R + ec);  // impl:268-275
    if (flip && idx != cfg.action_size - 1) {                // impl:700-720 (the noop index is perspective-invariant)
        const int start = floor_div(idx, cfg.mpa), off = floor_mod(idx, cfg.mpa);  // impl:369-383
        const int sr = floor_div(start, cfg.C), sc = floor_mod(start, cfg.C);
        const int tr = off >= cfg.R ? sr : off, tc = off >= cfg.R ? off - cfg.R : sc;
        const int fsr = cfg.R - 1 - sr, fsc = cfg.C - 1 - sc, fer = cfg.R - 1 - tr, fec = cfg.C - 1 - tc;  // impl:687-695
        idx = (fsr * cfg.C + fsc) * cfg.mpa + (fer != fsr ? fer : cfg.R + fec);
    }
    return idx;
}

// flat spatial index in the mover's frame: maenv:685 (unravel; out of range raises) + impl:316-347 + impl:700-720.
// Targets on the board take the direct route (identical to the reference's index arithmetic there); everything else
// goes through the reference's unchecked 1D aliasing above.
__device__ __forceinline__ Move decode_spatial(const DevConfig &cfg, int action, int flip)
{
    Move mv{0, 0, 0, 0, 0, 0, false, true};
    if (action < 0 || action >= cfg.N * cfg.A) return mv;
    const int cell = fast_div(action, cfg.magic_A), ch = action - cell * cfg.A;
    const int r = fast_div(cell, cfg.magic_C), c = cell - r * cfg.C;
    const int mr = cfg.R - 1, mc = cfg.C - 1;
    int er = r, ec = c;
    if (ch < mr) er = r + ch + 1;
    else if (ch < 2 * mr) er = r - (ch - mr + 1);
    else if (ch < 2 * mr + mc) ec = c + (ch - 2 * mr + 1);
    else ec = c - (ch - 2 * mr - mc + 1);  // impl:331-333: the noop channel lands here too (ec = c - C)
    if (er < 0 || er >= cfg.R || ec < 0 || ec >= cfg.C) return decode_1d(cfg, alias_spatial_1d(&cfg, cell, r, er, ec, flip));
    mv.sr = flip ? cfg.R - 1 - r : r;
    mv.sc = flip ? cfg.C - 1 - c : c;
    mv.er = flip ? cfg.R - 1 - er : er;
    mv.ec = flip ? cfg.C - 1 - ec : ec;
    mv.start = mv.sr * cfg.C + mv.sc;
    mv.end = mv.er * cfg.C + mv.ec;
    mv.bad = false;
    return mv;
}

enum StepStatus { STEP_ILLEGAL = 0, STEP_UNCHANGED = 1, STEP_NOOP_LOSS = 2, STEP_MOVED = 3 };

// impl:726-798 on the compact state (warp-uniform)
__device__ __forceinline__ bool move_is_legal(const DevConfig &cfg, const WarpMem &m, const Aux &a, const Move &mv,
                                              bool allow_osc)
{
    if (a.over || mv.bad) return false;
    const int me = a.to_move;
    const uint32_t sb = m.board[mv.start], eb = m.board[mv.end];
    const int rank = sb & CELL_RANK;
    if (rank == 0 || rank > SP_MARSHAL || int((sb >> 4) & 1) != me) return false;
    if (eb & CELL_OBST) return false;
    if ((eb & CELL_RANK) != 0 && int((eb >> 4) & 1) == me) return false;
    const int sr = mv.sr, sc = mv.sc, er = mv.er, ec = mv.ec;
    if ((sr != er) == (sc != ec)) return false;  // diagonal or zero-length
    if (!allow_osc && a.rcode[me] == 3 && a.rto[me] == mv.start && a.rfrom[me] == mv.end && (eb & CELL_RANK) == 0)
        return false;  // impl:771-777
    const int delta = sr != er ? (er - sr) * cfg.C : (ec - sc);
    const int dist = sr != er ? (er > sr ? er - sr : sr - er) : (ec > sc ? ec - sc : sc - ec);
    if (rank == SP_SCOUT) {
        const int stepv = delta / dist;
        for (int t = 1, cell = mv.start + stepv; t < dist; ++t, cell += stepv)
            if (m.board[cell] != 0) return false;  // impl:779-792
    } else if (dist > 1) {
        return false;  // impl:794
    }
    return true;
}

// records one captured piece (impl:999-1009) in the capture list; lanes search entries in parallel
// A capture that does not fit (count beyond 8 in one entry, or more distinct entries than the list holds: neither can
// happen in games played from a variant's own setups, whose list is sized 2 x pieces) is NOT dropped silently: the
// game's sticky overflow flag is raised and the step reports it (`illegal` = 2), because the reference's dense int64
// counters (impl:999-1009) would have kept counting.
template <class GT>
__device__ __forceinline__ void add_capture_inl(const DevConfig &cfg, const WarpMem &m, Aux &a, int cell, int owner, int type)
{
    const uint32_t key = cap_key(cell, owner, type);
    const int lane = GT::lane();
    int hit = -1;
    for (int e = lane; e < a.ncap; e += GT::L)
        if ((uint32_t(m.cap[e]) & 0x1fffu) == key) hit = e;
    const bool vote = GT::any(hit >= 0);
    if (vote) {
        const bool full = GT::any(hit >= 0 && (m.cap[hit] >> 13) >= 7);
        if (full) a.overflow = 1;
        else if (hit >= 0) m.cap[hit] = uint16_t(m.cap[hit] + (1u << 13));
    } else if (a.ncap < cfg.cap_stride) {
        if (lane == 0) m.cap[a.ncap] = uint16_t(key);
        a.ncap += 1;
    } else {
        a.overflow = 1;
    }
    GT::sync();
}

// Out-of-line entry (attacks are 2-4 % of moves): arguments and result by value so that the caller's
// Aux stays in registers.
// Returns the new entry count, or -1 - count when the capture did not fit.
template <class GT>
static __device__ __noinline__ int add_capture(const DevConfig *cfg, uint16_t *cap, int ncap, int cell, int owner, int type)
{
    WarpMem m{};
    m.cap = cap;
    Aux a{};
    a.ncap = ncap;
    add_capture_inl<GT>(*cfg, m, a, cell, owner, type);
    return a.overflow ? -1 - a.ncap : a.ncap;
}

// impl:897-1028: applies a decoded move for the player to move.  The opponent-stuck and max-turn
// checks (impl:1031-1043) need the next player's move list and are done by the caller.
template <class GT>
__device__ __forceinline__ StepStatus apply_move(const DevConfig &cfg, const WarpMem &m, Aux &a, const Move &mv,
                                                 bool allow_osc, int &attack)
{
    attack = 0;
    const int me = a.to_move, player = me == 0 ? 1 : -1;
    if (mv.noop) {  // impl:809-814: a noop is legal only when nothing else is
        if (mv.bad) return STEP_ILLEGAL;
        if (a.over) { a.to_move ^= 1; return STEP_UNCHANGED; }  // impl:907-909
        // the caller runs gen_moves for a noop first and passes mv.bad = true when moves exist, so
        // reaching this point means the player is stuck.
        a.turn += 1;  // impl:912-920
        a.over = 1;
        a.winner = -player;
        a.to_move ^= 1;
        return STEP_NOOP_LOSS;
    }
    if (!move_is_legal(cfg, m, a, mv, allow_osc)) return STEP_ILLEGAL;

    const uint32_t sb = m.board[mv.start], eb = m.board[mv.end];
    const int rank = sb & CELL_RANK, defender = eb & CELL_RANK;
    const int sr = mv.sr, er = mv.er;
    const int dist = sr != er ? (er > sr ? er - sr : sr - er)
                              : (mv.end > mv.start ? mv.end - mv.start : mv.start - mv.end);
    a.turn += 1;
    uint32_t new_start = 0, new_end;  // still flags at start/end are cleared for both sides (impl:939-941)
    bool wins = false, tie = false;
    if (defender == 0) {  // impl:955-964
        const uint32_t revealed = dist > 1 ? CELL_REVEALED : (sb & CELL_REVEALED);
        new_end = uint32_t(rank) | (uint32_t(me) << 4) | revealed;
    } else {  // impl:966-995
        attack = 1;
        if (rank == SP_MINER && defender == SP_BOMB) wins = true;
        else if (rank == SP_SPY && defender == SP_MARSHAL) wins = true;
        else if (defender == SP_FLAG) { a.over = 1; a.winner = player; wins = true; }
        else if (defender != SP_BOMB) { tie = rank == defender; wins = rank > defender; }
        if (wins) new_end = uint32_t(rank) | (uint32_t(me) << 4) | CELL_REVEALED;
        else if (tie) new_end = 0;
        else new_end = (eb & (CELL_RANK | CELL_OWNER)) | CELL_REVEALED;
    }
    GT::sync();
    if (GT::lane() == 0) { m.board[mv.start] = uint8_t(new_start); m.board[mv.end] = uint8_t(new_end); }
    GT::sync();
    if (defender != 0) {  // impl:999-1009
        if (!wins) {
            const int n = add_capture<GT>(&cfg, m.cap, a.ncap, mv.end, me, rank);
            if (n < 0) { a.overflow = 1; a.ncap = -1 - n; } else a.ncap = n;
        }
        if (wins || tie) {
            const int n = add_capture<GT>(&cfg, m.cap, a.ncap, mv.end, me ^ 1, defender);
            if (n < 0) { a.overflow = 1; a.ncap = -1 - n; } else a.ncap = n;
        }
    }
    // impl:1013-1028: the mover's recent-move record is rebuilt from scratch
    if (defender == 0) {
        const bool onto_came_from = a.rfrom[me] == mv.end;
        const bool from_next_illegal = a.rto[me] == mv.start && a.rcode[me] == 2;
        a.rcode[me] = onto_came_from ? (from_next_illegal ? 3 : 2) : 1;
        a.rfrom[me] = mv.start;
        a.rto[me] = mv.end;
    } else {
        a.rfrom[me] = NO_CELL; a.rto[me] = NO_CELL; a.rcode[me] = 0;
    }
    a.to_move ^= 1;
    return STEP_MOVED;
}

// impl:1029-1043, the rest of a step after apply_move returned STEP_MOVED for `mover`: the next player's move sets in
// m.moves, the opponent-stuck win and the turn limit.  Returns whether the next player has a move.  Used by the search
// kernels (sx_expand.cu, sx_playout.cu); the fused kernel keeps its own copy, which also serves viewers other than the
// player to move and the terminal re-generation of its outputs.
template <int K, class GT, bool CM>
__device__ __forceinline__ bool after_move(const DevConfig &cfg, const WarpMem &m, Aux &a, int mover)
{
    const bool any = gen_moves<K, GT, CM>(cfg, m, a, a.to_move, false);
    if (!any && !a.over) { a.over = 1; a.winner = mover == 0 ? 1 : -1; }  // impl:1031-1036
    if (a.turn >= a.max_turns && !a.over) { a.over = 1; a.invalid = 1; }  // impl:1040-1043
    return any;
}

// stages game b's board (padding included) and, with scap non-null, its capture list in shared memory (one warp);
// returns its packed aux words
__device__ __forceinline__ uint4 load_game(const DevConfig &cfg, const uint8_t *board, const int16_t *aux, const uint16_t *cap,
                                           long long b, uint8_t *sboard, uint16_t *scap)
{
    const int lane = threadIdx.x & 31;
    const uint32_t *gb = reinterpret_cast<const uint32_t *>(board + b * cfg.board_stride);
    for (int w = lane; w < (cfg.board_stride >> 2); w += 32) reinterpret_cast<uint32_t *>(sboard)[w] = gb[w];
    if (scap) {
        const uint32_t *gc = reinterpret_cast<const uint32_t *>(cap + b * cfg.cap_stride);
        for (int w = lane; w < (cfg.cap_stride >> 1); w += 32) reinterpret_cast<uint32_t *>(scap)[w] = gc[w];
    }
    return *reinterpret_cast<const uint4 *>(aux + b * 8);
}

__device__ __forceinline__ void unpack(uint4 aw, Aux &a)
{
    const uint32_t w[4] = {aw.x, aw.y, aw.z, aw.w};
    aux_unpack(w, a);
}

// writes the game staged in shared memory (board with padding, capture list) and the packed aux words `aw` to row `row`
// of a state (one warp; the inverse of load_game)
__device__ __forceinline__ void store_game(const DevConfig &cfg, const WarpMem &m, const uint32_t aw[4], uint8_t *board,
                                           int16_t *aux, uint16_t *cap, long long row)
{
    const int lane = threadIdx.x & 31;
    uint32_t *gb = reinterpret_cast<uint32_t *>(board + row * cfg.board_stride);
    for (int w = lane; w < (cfg.board_stride >> 2); w += 32) gb[w] = reinterpret_cast<const uint32_t *>(m.board)[w];
    uint32_t *gc = reinterpret_cast<uint32_t *>(cap + row * cfg.cap_stride);
    for (int w = lane; w < (cfg.cap_stride >> 1); w += 32) gc[w] = reinterpret_cast<const uint32_t *>(m.cap)[w];
    if (lane == 0) *reinterpret_cast<uint4 *>(aux + row * 8) = make_uint4(aw[0], aw[1], aw[2], aw[3]);
}

// the six scalars of a step that left the game in `a`, as sx_fused_kernel writes them (one lane); the caller says
// whether the game is done and what `illegal` holds
__device__ __forceinline__ void store_step_scalars(const sx_outputs &o, long long row, const Aux &a, bool done, int illegal)
{
    const int win = a.winner;
    if (o.done) o.done[row] = done ? 1 : 0;
    if (o.winner) o.winner[row] = int8_t(done ? win : 0);
    if (o.ending_invalid) o.ending_invalid[row] = (done && a.invalid) ? 1 : 0;
    if (o.illegal) o.illegal[row] = uint8_t(illegal);
    if (o.reward) o.reward[row] = (done && !a.invalid) ? float(win) : 0.0f;  // maenv:777-801
    if (o.player) o.player[row] = a.to_move == 0 ? 1 : -1;
}

// ---- setups / reset (impl:213-249, util:13-53, util:241-319) ---------------------------------------
// own_map[i], i < setup_len: piece code at own-frame cell i (row-major over the usable rows).
template <class GT>
__device__ __forceinline__ void place_side(const DevConfig &cfg, const WarpMem &m, const uint8_t *own_map, int side)
{
    for (int i = GT::lane(); i < cfg.setup_len; i += GT::L) {
        const int code = own_map[i];
        if (code == 0) continue;
        const int r = i / cfg.C, c = i - r * cfg.C;
        int cell;
        if (side == 0) cell = i;                                                    // impl:220
        else if (cfg.p2_rot180) cell = cfg.N - 1 - i;                                // impl:221
        else cell = (cfg.R - 1 - r) * cfg.C + c;                                     // util:263-273 net effect
        m.board[cell] = uint8_t(uint32_t(code) | (uint32_t(side) << 4) | CELL_STILL);  // impl:224-243
    }
}

template <class GT>
__device__ __forceinline__ void shuffle_side(const DevConfig &cfg, const WarpMem &m, uint8_t *perm, uint8_t *own_map,
                                             uint2 key, uint64_t gid, uint32_t episode, int side, uint32_t attempt)
{
    // util:13-30: shuffle the usable cells, then deal pieces in piece-code order
    const int n = cfg.setup_len;
    for (int i = GT::lane(); i < n; i += GT::L) { perm[i] = uint8_t(i); own_map[i] = 0; }
    GT::sync();
    if (GT::lane() == 0) {
        uint4 rnd = make_uint4(0, 0, 0, 0);
        int have = 0;
        uint32_t block = 0;
        for (int i = n - 1; i >= 1; --i) {
            if (have == 0) {
                rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SHUFFLE + uint32_t(side) + 2 * block + 64u * attempt, episode), key);
                have = 4;
                ++block;
            }
            const uint32_t u = have == 4 ? rnd.x : have == 3 ? rnd.y : have == 2 ? rnd.z : rnd.w;
            --have;
            const int j = int(__umulhi(u, uint32_t(i + 1)));
            const uint8_t t = perm[i]; perm[i] = perm[j]; perm[j] = t;
        }
        for (int k = 0; k < cfg.n_pieces; ++k) own_map[perm[k]] = cfg.piece_seq[k];
    }
    GT::sync();
}

struct ResetSource {
    const uint8_t *setups;     // [n_setups][setup_len] or null
    int n_setups;
    const int32_t *setup_idx;  // [2] rows for this env, or null = draw
    bool shuffle;
    // Which draw: the Philox counter holds (global env id, stream + 64 * attempt, rng_episode).  rng_episode is the game's
    // episode number, 0 for every game with same_start_pos_everytime (maenv:352-354), or the PREVIOUS episode's number
    // when the game repeats the last setup from the other side (maenv:530-534); attempt counts re-draws of an unplayable
    // setup, so that re-drawing never disturbs the episode numbering.
    uint32_t rng_episode, attempt;
    bool other_side;           // maenv:530-534: last initial state as player -1 sees it (impl:646-675), player -1 moves first
};

template <class GT>
__device__ __forceinline__ void reset_game_inl(const DevConfig &cfg, const WarpMem &m, Aux &a, const ResetSource &src,
                                               uint2 key, uint64_t gid)
{
    const int lane = GT::lane();
    GT::sync();
    for (int i = lane; i < cfg.board_stride; i += GT::L) m.board[i] = (i < cfg.N && cfg.obstacles[i]) ? uint8_t(CELL_OBST) : uint8_t(0);
    GT::sync();
    const uint32_t episode = a.episode;
    if (src.shuffle || src.setups == nullptr) {
        uint8_t *perm = m.scratch, *own_map = m.scratch + cfg.setup_len;
        for (int side = 0; side < 2; ++side) {
            shuffle_side<GT>(cfg, m, perm, own_map, key, gid, src.rng_episode, side, src.attempt);
            place_side<GT>(cfg, m, own_map, side);
            GT::sync();
        }
    } else {
        int i0, i1;
        if (src.setup_idx) { i0 = src.setup_idx[0]; i1 = src.setup_idx[1]; }
        else {
            const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_RESET + 64u * src.attempt, src.rng_episode), key);
            i0 = int(__umulhi(rnd.x, uint32_t(src.n_setups)));  // util:313-314: two independent uniform draws
            i1 = int(__umulhi(rnd.y, uint32_t(src.n_setups)));
        }
        place_side<GT>(cfg, m, src.setups + size_t(i0) * cfg.setup_len, 0);
        place_side<GT>(cfg, m, src.setups + size_t(i1) * cfg.setup_len, 1);
    }
    GT::sync();
    if (src.other_side) {  // impl:646-675 on the fresh board: rotate 180 degrees, swap the owners
        for (int i = lane; 2 * i < cfg.N; i += GT::L) {
            const int j = cfg.N - 1 - i;
            uint32_t x = m.board[i], y = m.board[j];
            if (x & CELL_RANK) x ^= CELL_OWNER;
            if (y & CELL_RANK) y ^= CELL_OWNER;
            if (i == j) m.board[i] = uint8_t(x);
            else { m.board[i] = uint8_t(y); m.board[j] = uint8_t(x); }
        }
        GT::sync();
    }
    a.turn = 0;
    a.max_turns = cfg.max_turns;  // impl:247
    a.over = 0; a.invalid = 0; a.winner = 0;
    a.to_move = src.other_side ? 1 : 0;  // maenv:546 / maenv:534
    a.rfrom[0] = a.rfrom[1] = NO_CELL;
    a.rto[0] = a.rto[1] = NO_CELL;
    a.rcode[0] = a.rcode[1] = 0;
    a.ncap = 0;
    a.overflow = 0;
    a.episode = episode + 1;
}

// Out-of-line entry: re-sets the game staged in the warp slice at `warp_base`, returns the packed aux words.
// `draw` packs attempt (bits 0-7), "other side" (bit 8) and "shuffle" (bit 9).
template <class GT>
static __device__ __noinline__ uint4 reset_game(const DevConfig *cfg, uint8_t *warp_base, const uint8_t *setups, int n_setups,
                                         const int32_t *setup_idx, uint32_t draw, uint2 key, uint64_t gid, uint32_t episode,
                                         uint32_t rng_episode)
{
    WarpMem m;
    carve_warp(*cfg, warp_base, &m);
    Aux a{};
    a.episode = episode;
    const ResetSource src{setups, n_setups, setup_idx, (draw & 512u) != 0, rng_episode, draw & 255u, (draw & 256u) != 0};
    reset_game_inl<GT>(*cfg, m, a, src, key, gid);
    uint32_t w[4];
    aux_pack(a, w);
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// Curriculum start (util:373-387, maenv:519-527): the game staged at `warp_base` becomes a uniformly drawn entry of a table
// of compact states; the turn counter restarts at 0 with the configured max_turns (util:382-383), the player to move is
// drawn uniformly (maenv:523), the markers of recent moves and the captured pieces stay as the entry has them.  Same
// Philox stream as a setup draw (RNG_RESET, attempt number, episode).  Returns the packed aux words.
template <class GT>
static __device__ __noinline__ uint4 reset_from_table(const DevConfig *cfg, uint8_t *warp_base, const uint8_t *t_board,
                                                      const int16_t *t_aux, const uint16_t *t_cap, uint32_t n_states,
                                                      uint32_t attempt, uint2 key, uint64_t gid, uint32_t episode,
                                                      uint32_t rng_episode, int32_t *index_out)
{
    WarpMem m;
    carve_warp(*cfg, warp_base, &m);
    const int lane = GT::lane();
    const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_RESET + 64u * attempt, rng_episode), key);
    const size_t idx = __umulhi(rnd.x, n_states);
    GT::sync();
    const uint32_t *gb = reinterpret_cast<const uint32_t *>(t_board + idx * cfg->board_stride);
    const uint32_t *gc = reinterpret_cast<const uint32_t *>(t_cap + idx * cfg->cap_stride);
    for (int i = lane; i < (cfg->board_stride >> 2); i += GT::L) reinterpret_cast<uint32_t *>(m.board)[i] = gb[i];
    for (int i = lane; i < (cfg->cap_stride >> 1); i += GT::L) reinterpret_cast<uint32_t *>(m.cap)[i] = gc[i];
    const uint4 aw = *reinterpret_cast<const uint4 *>(t_aux + idx * 8);
    const uint32_t w0[4] = {aw.x, aw.y, aw.z, aw.w};
    Aux a;
    aux_unpack(w0, a);
    a.turn = 0;
    a.max_turns = cfg->max_turns;
    a.to_move = int(rnd.y & 1u);
    a.episode = episode + 1;
    if (index_out != nullptr && lane == 0) *index_out = int32_t(idx);
    GT::sync();
    uint32_t w[4];
    aux_pack(a, w);
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// ---- observation tiles (impl:1232-1397 + maenv:499-508) ---------------------------------------------
// Channel map of the partial (impl:1306-1332) and full (impl:1200-1227) observations.
struct ObsMap {
    int channels, own_true, enemy_true /* -1 = absent */, own_po, enemy_po, obstacle, own_recent, enemy_recent,
        own_cap, enemy_cap, own_still, enemy_still;
};
__device__ __forceinline__ ObsMap po_map() { return ObsMap{67, 0, -1, 12, 25, 38, 39, 40, 41, 53, 65, 66}; }
__device__ __forceinline__ ObsMap fo_map() { return ObsMap{79, 0, 12, 24, 37, 50, 51, 52, 53, 65, 77, 78}; }
// the deprecated 'original' channel mode: one channel per state layer (impl:1126-1148 partial, impl:1048-1070 full)
__device__ __forceinline__ ObsMap po_map_original() { return ObsMap{32, 0, -1, 1, 2, 3, 4, 5, 6, 18, 30, 31}; }
__device__ __forceinline__ ObsMap fo_map_original() { return ObsMap{33, 0, 1, 5, 6, 2, 3, 4, 7, 19, 31, 32}; }

// Rows (cells) to skip at the start of a background image so that the copy's source is congruent mod 16 to a
// destination that is `a` words past a 16-byte boundary: the image is periodic in the cell, and a cell is
// `channels` words, so k cells shift the phase by k * channels words (67, 79 = 3 mod 4; 33 = 1 mod 4; 32 = 0).
__device__ __forceinline__ int align_rows(int channels, int a)
{
    const int c = channels & 3;
    return c == 3 ? ((4 - a) & 3) : c == 1 ? a : 0;
}

// The same for 16-bit observations, whose rows start at any even address: a cell is `channels` half-words, so k cells
// shift the phase by k * channels half-words mod 8, and a destination h half-words past a 16-byte boundary needs
// k * channels = h (mod 8).  For the odd channel counts (67, 79, 33) k = h * channels mod 8 solves it (an odd c has
// c * c = 1 mod 8), so up to 7 skipped cells (carve_tile: 7 extra image rows).  32 channels are 64 bytes per cell:
// no skip changes the phase, and none is needed, since every game row of such a tensor starts 16-byte aligned.
__host__ __device__ inline int align_cells16(int channels, int h) { return (channels & 1) ? ((h * channels) & 7) : 0; }

// Observation element type T: float (the LUT values as they are) or uint16_t, the bfloat16 / float16 bit pattern that
// sx_config_create has put into the low half of each LUT word (sx_config_desc::obs_dtype).
template <class T> __device__ __forceinline__ T obs_value(float lut_word);
template <> __device__ __forceinline__ float obs_value<float>(float lut_word) { return lut_word; }
template <> __device__ __forceinline__ uint16_t obs_value<uint16_t>(float lut_word) { return uint16_t(__float_as_uint(lut_word)); }

// extra cells at the end of a background image, for the alignment skip of align_rows / align_cells16
template <class T> __host__ __device__ constexpr int bg_extra_cells() { return sizeof(T) == 4 ? 3 : 7; }

// fills a tile with what an empty board looks like after normalisation
template <class T = float>
static __device__ __noinline__ void fill_background(const DevConfig &cfg, T *tile, const ObsMap om, int first, int stride,
                                                    int cells)
{
    const int total = cells * om.channels;
#pragma unroll 1
    for (int i = first; i < total; i += stride) {
        const int ch = i % om.channels;
        float v = cfg.unit_lut[0];
        if (ch == om.own_recent || ch == om.enemy_recent) v = cfg.recent_lut[3];
        else if (ch >= om.own_cap && ch < om.own_cap + 12) v = cfg.cap_lut[(ch - om.own_cap) * 9];
        else if (ch >= om.enemy_cap && ch < om.enemy_cap + 12) v = cfg.cap_lut[(ch - om.enemy_cap) * 9];
        else if (cfg.original_channels) {  // rank planes hold "no piece" instead of a one-hot zero
            if (ch == om.own_true || ch == om.enemy_true) v = cfg.rank_lut[0];
            else if (ch == om.own_po || ch == om.enemy_po) v = cfg.po_rank_lut[0];
        }
        tile[i] = obs_value<T>(v);
    }
}

// One game's background copy of a 16-bit observation of `elems` elements to `g`: the image row that makes the copy's
// source congruent to g mod 16 is chosen, so the body leaves as one TMA bulk copy.
template <class GT>
__device__ __forceinline__ void emit_obs16(uint16_t *g, const uint16_t *bg, int channels, int elems)
{
    const int k = align_cells16(channels, int((reinterpret_cast<uintptr_t>(g) >> 1) & 7));
    emit_tile16<GT>(reinterpret_cast<uint8_t *>(g), reinterpret_cast<const uint8_t *>(bg + k * channels), elems * 2);
}

// Writes the sparse, state-dependent entries of observer `me`'s observation on top of the background
// image at `tile` (global memory).
// ORIG = the deprecated 'original' channel mode: rank planes carry the normalised rank instead of one-hot groups.
template <int K, class GT, bool ORIG = false, class T = float>
__device__ __forceinline__ void patch_obs(const DevConfig &cfg, const WarpMem &m, const Aux &a, T *tile,
                                          const ObsMap om, int me)
{
    const int lane = GT::lane(), flip = me, CH = om.channels;
    const T one = obs_value<T>(cfg.unit_lut[1]);
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p < cfg.N) {
            const uint32_t b = m.board[view(p, flip, cfg.N)];
            T *cell = tile + p * CH;
            if (b & CELL_OBST) *(cell + om.obstacle) = one;
            const int rank = b & CELL_RANK;
            if (rank) {
                const int po = (b & CELL_REVEALED) ? rank : SP_UNKNOWN;
                const bool own = int((b >> 4) & 1) == me;
                if (ORIG) {  // impl:1178-1195 / impl:1102-1121 + maenv:499-508
                    if (own || om.enemy_true >= 0)
                        *(cell + (own ? om.own_true : om.enemy_true)) = obs_value<T>(cfg.rank_lut[rank]);
                    *(cell + (own ? om.own_po : om.enemy_po)) = obs_value<T>(cfg.po_rank_lut[po]);
                    if (b & CELL_STILL) *(cell + (own ? om.own_still : om.enemy_still)) = one;
                } else if (own) {
                    *(cell + om.own_true + rank - 1) = one;
                    *(cell + om.own_po + po - 1) = one;
                    if (b & CELL_STILL) *(cell + om.own_still) = one;
                } else {
                    if (om.enemy_true >= 0) *(cell + om.enemy_true + rank - 1) = one;
                    *(cell + om.enemy_po + po - 1) = one;
                    if (b & CELL_STILL) *(cell + om.enemy_still) = one;
                }
            }
        }
    }
    if (lane < 4) {  // recent-move squares: lanes 0/1 own from/to, lanes 2/3 enemy from/to
        const int who = (lane < 2) ? me : (me ^ 1);
        const int cell_abs = (lane & 1) ? a.rto[who] : a.rfrom[who];
        const int code = (lane & 1) ? -a.rcode[who] : 1;
        if (cell_abs != NO_CELL)
            *(tile + view(cell_abs, flip, cfg.N) * CH + (lane < 2 ? om.own_recent : om.enemy_recent)) =
                obs_value<T>(cfg.recent_lut[code + 3]);
    }
    for (int e = lane; e < a.ncap; e += GT::L) {
        const uint32_t ent = m.cap[e];
        const int cell_abs = ent & 0xff, owner = (ent >> 8) & 1, type0 = (ent >> 9) & 15, count = int(ent >> 13) + 1;
        *(tile + view(cell_abs, flip, cfg.N) * CH + (owner == me ? om.own_cap : om.enemy_cap) + type0) =
            obs_value<T>(cfg.cap_lut[type0 * 9 + count]);
    }
}

// position of the n-th (0-based) set bit of a 64-bit set that has more than n bits: six popcount-guided halvings
// (one __fns per 32-bit half costs about twice as many instructions)
__device__ __forceinline__ int nth_set_bit64(uint2 bits, int n)
{
    int pos = 0;
    uint32_t x = bits.x;
    const int c0 = __popc(bits.x);
    if (n >= c0) { n -= c0; x = bits.y; pos = 32; }
#pragma unroll
    for (int w = 16; w >= 1; w >>= 1) {
        const int c = __popc(x & ((1u << w) - 1u));
        if (n >= c) { n -= c; x >>= w; pos += w; }
    }
    return pos;
}

// ---- uniform draw over the generated moves (replaces maenv:830-834) ----------------------------------
// Order = ascending flat spatial index (cell, then channel).
template <int K, class GT>
__device__ __forceinline__ int sample_move(const DevConfig &cfg, const WarpMem &m, bool any_moves, uint32_t rnd)
{
    if (!any_moves) return cfg.A - 1;  // the noop entry [0,0,A-1]
    const int lane = GT::lane();
    int mine = 0;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p < cfg.N) {
            const uint2 bits = m.moves[p];
            mine += __popc(bits.x) + __popc(bits.y);
        }
    }
    int incl = mine;
#pragma unroll
    for (int off = 1; off < GT::L; off <<= 1) {
        const int v = GT::shfl_up(incl, off);
        if (lane >= off) incl += v;
    }
    const int total = GT::shfl(incl, GT::L - 1);
    const int t = int(__umulhi(rnd, uint32_t(total)));
    int action = 0;
    const bool owner = t >= incl - mine && t < incl;
    if (owner) {
        int left = t - (incl - mine);
#pragma unroll 1
        for (int k = 0; k < K; ++k) {
            const int p = lane * K + k;
            const uint2 bits = p < cfg.N ? m.moves[p] : make_uint2(0, 0);
            const int c0 = __popc(bits.x), c1 = __popc(bits.y);
            if (left < c0 + c1) {
                uint32_t w = left < c0 ? bits.x : bits.y;
                int skip = left < c0 ? left : left - c0;
#pragma unroll 1
                for (; skip > 0; --skip) w &= w - 1;
                action = p * cfg.A + (left < c0 ? 0 : 32) + __ffs(w) - 1;
                break;
            }
            left -= c0 + c1;
        }
    }
    const uint32_t who = GT::ballot(owner);
    return GT::shfl(action, __ffs(who) - 1);
}

// ---- per-warp helpers of the search kernels (sx_expand.cu, sx_playout.cu, sx_search.cu, sx_guided.cu; Grp<1>) ------

// the moves in m.moves of this lane's K cells
template <int K>
__device__ __forceinline__ int lane_moves(const DevConfig &cfg, const WarpMem &m)
{
    const int lane = threadIdx.x & 31;
    int mine = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p < cfg.N) mine += __popc(m.moves[p].x) + __popc(m.moves[p].y);
    }
    return mine;
}

// `mine`: lane_moves; `incl`: its inclusive prefix sum over the warp, so this lane's moves are numbers
// incl - mine .. incl - 1 of the ascending list.  Returns the warp's total.
template <int K>
__device__ __forceinline__ int lane_move_scan(const DevConfig &cfg, const WarpMem &m, int &mine, int &incl)
{
    const int lane = threadIdx.x & 31;
    mine = lane_moves<K>(cfg, m);
    incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(FULL, incl, d);
        if (lane >= d) incl += v;
    }
    return __shfl_sync(FULL, incl, 31);
}

// fn(action) for each move of this lane's K cells in m.moves, in ascending flat spatial index
template <int K, class F>
__device__ __forceinline__ void for_each_lane_move(const DevConfig &cfg, const WarpMem &m, F fn)
{
    const int lane = threadIdx.x & 31;
#pragma unroll 1
    for (int k = 0; k < K; ++k) {
        const int p = lane * K + k;
        if (p >= cfg.N) break;
#pragma unroll 1
        for (int h = 0; h < 2; ++h)
            for (uint32_t w = h ? m.moves[p].y : m.moves[p].x; w; w &= w - 1) fn(p * cfg.A + h * 32 + __ffs(w) - 1);
    }
}

// the warp's largest (best, best_j) by score, the lowest index on a tie, on every lane; best_j < 0: the lane has none
__device__ __forceinline__ void warp_argmax(float &best, int &best_j)
{
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ob = __shfl_xor_sync(FULL, best, d);
        const int oj = __shfl_xor_sync(FULL, best_j, d);
        if (oj >= 0 && (best_j < 0 || ob > best || (ob == best && oj < best_j))) { best = ob; best_j = oj; }
    }
}

// the next game of this block's range [blockIdx.x * per_block, + per_block) below num_envs for the calling warp, or -1
// once the range is handed out.  `claimed` is the block's __shared__ count of games handed out, zero before the first
// call.  Games differ a lot in length, so the warps of a block take them as they finish (claim_grid sizes the launch).
__device__ __forceinline__ long long claim_next(unsigned long long &claimed, long long per_block, long long num_envs)
{
    const long long first = (long long)blockIdx.x * per_block;
    const long long end = first + per_block < num_envs ? first + per_block : num_envs;
    long long b = 0;
    if ((threadIdx.x & 31) == 0) b = first + (long long)atomicAdd(&claimed, 1ull);
    b = __shfl_sync(FULL, b, 0);
    return b < end ? b : -1;
}

}  // namespace sx
