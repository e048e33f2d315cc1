// sx_toy.cuh -- the fused env step for the toy boards (at most 16 cells: Micro 3x4, Tiny 4x4), one THREAD per game.
//
// A 10x10 game keeps a warp busy; a 12-cell game does not: even with four games per warp (Grp<4>) the warp-level
// kernel spends ~1 000 issue slots per Micro game and is issue-bound at 0.4 of the HBM roofline.  Here the rules
// run with one game per thread -- the whole state is 48 bytes and lives in registers: board (16 cell bytes in four
// words), capture list (eight 16-bit entries in four words) and the aux word -- and the 32 consecutive games of a warp
// are then rendered cooperatively:
//   * mask: every thread marks its own game's moves in ONE shared-memory image of the warp's 32 mask rows (they are
//     contiguous in the output tensor), which leaves as a single TMA bulk copy;
//   * observations: each warp owns two shared-memory tiles that hold the background image; per game the lanes undo
//     the entries of the tile's previous game, lanes 0..N-1 add their cell's entries, lanes 16..27 the recent-move and
//     capture entries, and lane 0 hands the tile to the TMA engine (cp.async.bulk shared -> global).
// No sparse store ever goes to global memory, so nothing depends on L2 residency and any number of copies can be in
// flight.  Same rules, same Philox streams, same sampling order as the warp-level kernel (sx_kernels.cu), which still
// serves every other launch type of these variants (reset masks, 1D masks, player overrides, original channels) and
// the last num_envs % 32 games of a batch; tests/test_gpu_parity.py compares the two kernels game by game.
#pragma once

#include "sx_device.cuh"

namespace sx {
namespace toy {

constexpr int GAMES = 32;        // games per warp-iteration = lanes
constexpr int STAGE_BYTES = 48;  // per game: board 16, capture list 16, recent-move info 8, pad

struct State {
    uint32_t b[4];  // board: one byte per cell (sx_device.cuh cell layout), cells 4j..4j+3 in word j
    uint32_t c[4];  // capture list: eight 16-bit entries
};

__device__ __forceinline__ uint32_t sel4(const uint32_t w[4], int j) { return j == 0 ? w[0] : j == 1 ? w[1] : j == 2 ? w[2] : w[3]; }
__device__ __forceinline__ uint32_t cell_get(const State &s, int i) { return (sel4(s.b, i >> 2) >> ((i & 3) * 8)) & 0xffu; }
__device__ __forceinline__ void cell_set(State &s, int i, uint32_t v)
{
    const int j = i >> 2, sh = (i & 3) * 8;
    const uint32_t keep = ~(0xffu << sh), put = v << sh;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (j == k) s.b[k] = (s.b[k] & keep) | put;
}
__device__ __forceinline__ uint32_t cap_get(const State &s, int e) { return (sel4(s.c, e >> 1) >> ((e & 1) * 16)) & 0xffffu; }
__device__ __forceinline__ void cap_set(State &s, int e, uint32_t v)
{
    const int j = e >> 1, sh = (e & 1) * 16;
    const uint32_t keep = ~(0xffffu << sh), put = v << sh;
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (j == k) s.c[k] = (s.c[k] & keep) | put;
}

// occupancy bit sets of a position (bit = absolute cell)
struct Sets {
    uint32_t block[2];  // what player index 0 / 1 cannot step onto: own pieces and lakes
    uint32_t enemy[2];  // the opponent's pieces
    uint32_t mover[2];  // own pieces that can move (ranks 1..10, impl:420)
    uint32_t scout[2];
    uint32_t any;       // pieces and lakes
};

__device__ __forceinline__ Sets make_sets(const State &s)
{
    uint32_t piece[2] = {0, 0}, mover[2] = {0, 0}, scout[2] = {0, 0}, obst = 0;
#pragma unroll
    for (int p = 0; p < 16; ++p) {
        const uint32_t b = (s.b[p >> 2] >> ((p & 3) * 8)) & 0xffu;
        const uint32_t rank = b & CELL_RANK, o = (b >> 4) & 1u, bit = 1u << p;
        if (b & CELL_OBST) obst |= bit;
        if (rank) {
            if (o) piece[1] |= bit; else piece[0] |= bit;
            if (rank <= SP_MARSHAL) { if (o) mover[1] |= bit; else mover[0] |= bit; }
            if (rank == SP_SCOUT) { if (o) scout[1] |= bit; else scout[0] |= bit; }
        }
    }
    Sets t;
    t.any = piece[0] | piece[1] | obst;
    t.block[0] = piece[0] | obst; t.block[1] = piece[1] | obst;
    t.enemy[0] = piece[1]; t.enemy[1] = piece[0];
    t.mover[0] = mover[0]; t.mover[1] = mover[1];
    t.scout[0] = scout[0]; t.scout[1] = scout[1];
    return t;
}

// a bit set in `me`'s frame: the 180-degree rotation is index reversal over the N cells
__device__ __forceinline__ uint32_t to_frame(uint32_t set, int flip, int N) { return flip ? (__brev(set) >> (32 - N)) : set; }

// Frame constants of a variant: cells that have a neighbour in each direction (bit = cell), computed once per thread.
struct Geometry {
    uint32_t has_down, has_up, has_right, has_left;  // +row, -row, +col, -col neighbour exists
};
__device__ __forceinline__ Geometry make_geometry(const DevConfig &cfg)
{
    Geometry g{0, 0, 0, 0};
#pragma unroll
    for (int p = 0; p < 16; ++p) {
        if (p < cfg.N) {
            const int r = fast_div(p, cfg.magic_C), c = p - r * cfg.C;
            if (r + 1 < cfg.R) g.has_down |= 1u << p;
            if (r > 0) g.has_up |= 1u << p;
            if (c + 1 < cfg.C) g.has_right |= 1u << p;
            if (c > 0) g.has_left |= 1u << p;
        }
    }
    return g;
}

// Move sets of a player, CHANNEL-major: bit p of a set = "the piece on cell p (the player's frame) may play this channel".
// The four one-square channels are exactly the four shifted occupancy sets move generation produces, so nothing is
// composed per cell; channels of two and more squares exist only with scouts on the board (none in the stock toy
// variants) and live in `far`, two 16-bit sets per word.  (Round 2: the cell-major mv[16] this replaces cost 189 static /
// 368 executed instructions per pass to compose and made the mask marking and the sampled-move select 16-way unrolled.)
struct MoveSets {
    // named members, not arrays: a run-time index into a register array makes the compiler keep the whole object in
    // local memory (the same trap as Aux's per-player pairs)
    uint32_t down, up, right, left;          // one-square channels 0, R-1, 2(R-1), 2(R-1)+C-1 (impl:292-311)
    uint32_t f0, f1, f2, f3, f4, f5, f6, f7;  // channel c (not a one-square channel): word c >> 1, half c & 1
    uint32_t any_far;                         // OR of f0..f7: 0 selects the fast paths
};
__device__ __forceinline__ void clear_sets(MoveSets &ms)
{
    ms.down = ms.up = ms.right = ms.left = 0;
    ms.f0 = ms.f1 = ms.f2 = ms.f3 = ms.f4 = ms.f5 = ms.f6 = ms.f7 = 0;
    ms.any_far = 0;
}
#define SX_TOY_FAR_WORD(ms, i, STMT)                                                                              \
    switch (i) {                                                                                                  \
    case 0: { uint32_t &w = ms.f0; STMT; } break;                                                                 \
    case 1: { uint32_t &w = ms.f1; STMT; } break;                                                                 \
    case 2: { uint32_t &w = ms.f2; STMT; } break;                                                                 \
    case 3: { uint32_t &w = ms.f3; STMT; } break;                                                                 \
    case 4: { uint32_t &w = ms.f4; STMT; } break;                                                                 \
    case 5: { uint32_t &w = ms.f5; STMT; } break;                                                                 \
    case 6: { uint32_t &w = ms.f6; STMT; } break;                                                                 \
    default: { uint32_t &w = ms.f7; STMT; } break;                                                                \
    }
// set / clear (cell p, channel ch) where ch is NOT a one-square channel
__device__ __forceinline__ void far_put(MoveSets &ms, int ch, int p)
{
    const uint32_t v = 1u << (p + 16 * (ch & 1));
    SX_TOY_FAR_WORD(ms, ch >> 1, w |= v)
    ms.any_far |= v;
}
__device__ __forceinline__ void far_clear(MoveSets &ms, int ch, int p)
{
    const uint32_t v = ~(1u << (p + 16 * (ch & 1)));
    SX_TOY_FAR_WORD(ms, ch >> 1, w &= v)
}
// the 16-bit channel set of cell p (bit = channel), the cell-major view the slow paths use
__device__ __forceinline__ uint32_t cell_channels(const DevConfig &cfg, const MoveSets &ms, int p)
{
    const int b1 = cfg.R - 1, b2 = 2 * b1, b3 = b2 + cfg.C - 1;
    uint32_t bits = ((ms.down >> p) & 1u) | (((ms.up >> p) & 1u) << b1) | (((ms.right >> p) & 1u) << b2) |
                    (((ms.left >> p) & 1u) << b3);
    const uint32_t far[8] = {ms.f0, ms.f1, ms.f2, ms.f3, ms.f4, ms.f5, ms.f6, ms.f7};
#pragma unroll
    for (int i = 0; i < 8; ++i)
        bits |= (((far[i] >> p) & 1u) << (2 * i)) | (((far[i] >> (p + 16)) & 1u) << (2 * i + 1));
    return bits;
}

// Valid moves of player index `me` in `me`'s frame (impl:400-517).  One-square moves of all pieces come from four shifts
// of the occupancy sets; scouts (absent from the stock toy variants, possible in custom ones) walk their rays in a
// rolled loop.  Returns the number of moves.
__device__ __forceinline__ int gen_moves(const DevConfig &cfg, const Geometry &geo, const State &s, const Aux &a, int me,
                                         bool allow_osc, MoveSets &ms)
{
    const int N = cfg.N, R = cfg.R, C = cfg.C;
    clear_sets(ms);
    if (a.over) return 0;  // impl:414
    const Sets t = make_sets(s);
    const int flip = me;
    const uint32_t block = to_frame(t.block[me], flip, N), movers = to_frame(t.mover[me], flip, N);
    const uint32_t scouts = to_frame(t.scout[me], flip, N);
    const int b1 = R - 1, b2 = 2 * b1, b3 = b2 + C - 1;
    // impl:492-512: a piece may step onto any neighbouring square that holds neither an own piece nor a lake
    const uint32_t walkers = movers & ~scouts;
    ms.down = walkers & geo.has_down & ~(block >> C);
    ms.up = walkers & geo.has_up & ~(block << C);
    ms.right = walkers & geo.has_right & ~(block >> 1);
    ms.left = walkers & geo.has_left & ~(block << 1);
    if (scouts != 0) {  // impl:426-490: slide until the edge, a lake or a piece; an enemy piece may be taken
        const uint32_t any = to_frame(t.any, flip, N), enemy = to_frame(t.enemy[me], flip, N);
#pragma unroll 1
        for (uint32_t left_scouts = scouts; left_scouts != 0; left_scouts &= left_scouts - 1) {
            const int p = __ffs(left_scouts) - 1;
            const int r = fast_div(p, cfg.magic_C), c = p - r * C;
            int n0 = 0, n1 = 0, n2 = 0, n3 = 0;
            for (int k = 1; r + k < R; ++k) { const int q = p + k * C; if ((any >> q) & 1u) { n0 += int((enemy >> q) & 1u); break; } ++n0; }
            for (int k = 1; r - k >= 0; ++k) { const int q = p - k * C; if ((any >> q) & 1u) { n1 += int((enemy >> q) & 1u); break; } ++n1; }
            for (int k = 1; c + k < C; ++k) { const int q = p + k; if ((any >> q) & 1u) { n2 += int((enemy >> q) & 1u); break; } ++n2; }
            for (int k = 1; c - k >= 0; ++k) { const int q = p - k; if ((any >> q) & 1u) { n3 += int((enemy >> q) & 1u); break; } ++n3; }
            const uint32_t bit = 1u << p;
            if (n0 > 0) ms.down |= bit;
            if (n1 > 0) ms.up |= bit;
            if (n2 > 0) ms.right |= bit;
            if (n3 > 0) ms.left |= bit;
#pragma unroll 1
            for (int k = 2; k <= n0; ++k) far_put(ms, k - 1, p);
#pragma unroll 1
            for (int k = 2; k <= n1; ++k) far_put(ms, b1 + k - 1, p);
#pragma unroll 1
            for (int k = 2; k <= n2; ++k) far_put(ms, b2 + k - 1, p);
#pragma unroll 1
            for (int k = 2; k <= n3; ++k) far_put(ms, b3 + k - 1, p);
        }
    }
    // the one move the two-square rule forbids (impl:439-445, 501-505), in `me`'s frame
    if (!allow_osc && a.rcode[me] == 3 && a.rto[me] != NO_CELL && a.rfrom[me] != NO_CELL &&
        (cell_get(s, a.rfrom[me]) & CELL_RANK) == 0) {
        const int sc_ = view(a.rto[me], flip, N), ec_ = view(a.rfrom[me], flip, N);
        const int sr = fast_div(sc_, cfg.magic_C), sc = sc_ - sr * C, er = fast_div(ec_, cfg.magic_C), ec = ec_ - er * C;
        if ((sr == er || sc == ec) && sc_ != ec_) {
            const int dir = sc == ec ? (er > sr ? 0 : 1) : (ec > sc ? 2 : 3);
            const int dist = sc == ec ? (er > sr ? er - sr : sr - er) : (ec > sc ? ec - sc : sc - ec);
            const uint32_t keep = ~(1u << sc_);
            if (dist == 1) {
                if (dir == 0) ms.down &= keep;
                else if (dir == 1) ms.up &= keep;
                else if (dir == 2) ms.right &= keep;
                else ms.left &= keep;
            } else {
                far_clear(ms, (dir == 0 ? 0 : dir == 1 ? b1 : dir == 2 ? b2 : b3) + dist - 1, sc_);
            }
        }
    }
    int total = __popc(ms.down) + __popc(ms.up) + __popc(ms.right) + __popc(ms.left);
    if (ms.any_far != 0)
        total += __popc(ms.f0) + __popc(ms.f1) + __popc(ms.f2) + __popc(ms.f3) + __popc(ms.f4) + __popc(ms.f5) + __popc(ms.f6) +
                 __popc(ms.f7);
    return total;
}

// impl:726-798 on the register state
__device__ __forceinline__ bool move_is_legal(const DevConfig &cfg, const State &s, const Aux &a, const Move &mv, bool allow_osc)
{
    if (a.over || mv.bad) return false;
    const int me = a.to_move;
    const uint32_t sb = cell_get(s, mv.start), eb = cell_get(s, mv.end);
    const int rank = sb & CELL_RANK;
    if (rank == 0 || rank > SP_MARSHAL || int((sb >> 4) & 1) != me) return false;
    if (eb & CELL_OBST) return false;
    if ((eb & CELL_RANK) != 0 && int((eb >> 4) & 1) == me) return false;
    const int sr = mv.sr, sc = mv.sc, er = mv.er, ec = mv.ec;
    if ((sr != er) == (sc != ec)) return false;
    if (!allow_osc && a.rcode[me] == 3 && a.rto[me] == mv.start && a.rfrom[me] == mv.end && (eb & CELL_RANK) == 0) return false;
    const int delta = sr != er ? (er - sr) * cfg.C : (ec - sc);
    const int dist = sr != er ? (er > sr ? er - sr : sr - er) : (ec > sc ? ec - sc : sc - ec);
    if (rank == SP_SCOUT) {
        const int stepv = delta / dist;
        for (int t = 1, cell = mv.start + stepv; t < dist; ++t, cell += stepv)
            if (cell_get(s, cell) != 0) return false;
    } else if (dist > 1) {
        return false;
    }
    return true;
}

// impl:999-1009 on the register capture list (eight entries)
__device__ __forceinline__ void add_capture(const DevConfig &cfg, State &s, Aux &a, int cell, int owner, int type)
{
    const uint32_t key = cap_key(cell, owner, type);
    int hit = -1;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const uint32_t ent = (s.c[e >> 1] >> ((e & 1) * 16)) & 0xffffu;
        if (e < a.ncap && (ent & 0x1fffu) == key) hit = e;
    }
    if (hit >= 0) {
        const uint32_t ent = cap_get(s, hit);
        if ((ent >> 13) < 7) cap_set(s, hit, ent + (1u << 13));
        else a.overflow = 1;  // see add_capture_inl (sx_device.cuh): never silent
    } else if (a.ncap < cfg.cap_stride) {
        cap_set(s, a.ncap, key);
        a.ncap += 1;
    } else {
        a.overflow = 1;
    }
}

// impl:897-1028 (same as apply_move of the warp-level kernel)
__device__ __forceinline__ StepStatus apply_move(const DevConfig &cfg, State &s, Aux &a, const Move &mv, bool allow_osc)
{
    const int me = a.to_move, player = me == 0 ? 1 : -1;
    if (mv.noop) {
        if (mv.bad) return STEP_ILLEGAL;
        if (a.over) { a.to_move ^= 1; return STEP_UNCHANGED; }
        a.turn += 1;
        a.over = 1;
        a.winner = -player;
        a.to_move ^= 1;
        return STEP_NOOP_LOSS;
    }
    if (!move_is_legal(cfg, s, a, mv, allow_osc)) return STEP_ILLEGAL;
    const uint32_t sb = cell_get(s, mv.start), eb = cell_get(s, mv.end);
    const int rank = sb & CELL_RANK, defender = eb & CELL_RANK;
    const int dist = mv.sr != mv.er ? (mv.er > mv.sr ? mv.er - mv.sr : mv.sr - mv.er)
                                    : (mv.end > mv.start ? mv.end - mv.start : mv.start - mv.end);
    a.turn += 1;
    uint32_t new_end;
    bool wins = false, tie = false;
    if (defender == 0) {
        const uint32_t revealed = dist > 1 ? CELL_REVEALED : (sb & CELL_REVEALED);
        new_end = uint32_t(rank) | (uint32_t(me) << 4) | revealed;
    } else {
        if (rank == SP_MINER && defender == SP_BOMB) wins = true;
        else if (rank == SP_SPY && defender == SP_MARSHAL) wins = true;
        else if (defender == SP_FLAG) { a.over = 1; a.winner = player; wins = true; }
        else if (defender != SP_BOMB) { tie = rank == defender; wins = rank > defender; }
        if (wins) new_end = uint32_t(rank) | (uint32_t(me) << 4) | CELL_REVEALED;
        else if (tie) new_end = 0;
        else new_end = (eb & (CELL_RANK | CELL_OWNER)) | CELL_REVEALED;
    }
    cell_set(s, mv.start, 0);
    cell_set(s, mv.end, new_end);
    if (defender != 0) {
        if (!wins) add_capture(cfg, s, a, mv.end, me, rank);
        if (wins || tie) add_capture(cfg, s, a, mv.end, me ^ 1, defender);
    }
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

// own_map: piece code per own-frame setup cell (at most 8 cells), one nibble... codes go up to 12, so one byte each
__device__ __forceinline__ void place_side(const DevConfig &cfg, State &s, unsigned long long own_map, int side)
{
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const uint32_t code = uint32_t(own_map >> (8 * i)) & 0xffu;
        if (i < cfg.setup_len && code != 0) {
            const int r = fast_div(i, cfg.magic_C), c = i - r * cfg.C;
            const int cell = side == 0 ? i : cfg.p2_rot180 ? cfg.N - 1 - i : (cfg.R - 1 - r) * cfg.C + c;  // impl:220-221, util:263-273
            cell_set(s, cell, code | (uint32_t(side) << 4) | CELL_STILL);
        }
    }
}

// util:13-30 with the warp-level kernel's Philox stream (shuffle_side in sx_device.cuh): draw k (0-based) of a side is
// word k % 4 of Philox block k / 4; a side of at most 8 setup cells needs at most 7 draws = two blocks
__device__ __forceinline__ unsigned long long shuffle_side(const DevConfig &cfg, uint2 key, uint64_t gid, uint32_t episode, int side,
                                                           uint32_t attempt)
{
    const int n = cfg.setup_len;
    uint32_t perm = 0x76543210u;  // perm[i] in nibble i
    const uint4 r0 = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SHUFFLE + uint32_t(side) + 64u * attempt, episode), key);
    uint4 r1 = make_uint4(0, 0, 0, 0);
    if (n > 5) r1 = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_SHUFFLE + uint32_t(side) + 2u + 64u * attempt, episode), key);
    const uint32_t draws[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
    int k = 0;
#pragma unroll
    for (int i = 7; i >= 1; --i) {
        if (i < n) {
            uint32_t u = draws[0];
#pragma unroll
            for (int d = 1; d < 8; ++d)
                if (k == d) u = draws[d];
            ++k;
            const int j = int(__umulhi(u, uint32_t(i + 1)));
            const uint32_t pi = (perm >> (4 * i)) & 15u, pj = (perm >> (4 * j)) & 15u;
            perm = (perm & ~(15u << (4 * i))) | (pj << (4 * i));
            perm = (perm & ~(15u << (4 * j))) | (pi << (4 * j));
        }
    }
    unsigned long long own_map = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q)
        if (q < cfg.n_pieces) own_map |= (unsigned long long)cfg.piece_seq[q] << (8 * ((perm >> (4 * q)) & 15u));
    return own_map;
}

__device__ __forceinline__ unsigned long long load_setup_row(const DevConfig &cfg, const uint8_t *row)
{
    unsigned long long own_map = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (i < cfg.setup_len) own_map |= (unsigned long long)row[i] << (8 * i);
    return own_map;
}

// impl:213-249 + the setup samplers (reset_game_inl of the warp-level kernel)
// rng_episode / attempt: see ResetSource (sx_device.cuh).  "Repeat from the other side" games do not come here (the launch
// goes to the warp-level kernel).
__device__ __forceinline__ void reset_game(const DevConfig &cfg, State &s, Aux &a, const uint8_t *setups, int n_setups, bool shuffle,
                                           uint2 key, uint64_t gid, uint32_t rng_episode, uint32_t attempt)
{
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t w = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (4 * j + k < cfg.N && cfg.obstacles[4 * j + k]) w |= CELL_OBST << (8 * k);
        s.b[j] = w;
    }
    const uint32_t episode = a.episode;
    if (shuffle || setups == nullptr) {
#pragma unroll 1
        for (int side = 0; side < 2; ++side) place_side(cfg, s, shuffle_side(cfg, key, gid, rng_episode, side, attempt), side);
    } else {
        const uint4 rnd = philox4x32_10(make_uint4(uint32_t(gid), uint32_t(gid >> 32), RNG_RESET + 64u * attempt, rng_episode), key);
        const int i0 = int(__umulhi(rnd.x, uint32_t(n_setups))), i1 = int(__umulhi(rnd.y, uint32_t(n_setups)));
        place_side(cfg, s, load_setup_row(cfg, setups + size_t(i0) * cfg.setup_len), 0);
        place_side(cfg, s, load_setup_row(cfg, setups + size_t(i1) * cfg.setup_len), 1);
    }
    a.turn = 0;
    a.max_turns = cfg.max_turns;
    a.over = 0; a.invalid = 0; a.winner = 0;
    a.to_move = 0;
    a.rfrom[0] = a.rfrom[1] = NO_CELL;
    a.rto[0] = a.rto[1] = NO_CELL;
    a.rcode[0] = a.rcode[1] = 0;
    a.ncap = 0;
    a.overflow = 0;
    a.episode = episode + 1;
}

// t-th move in ascending (cell, channel) order of the mover's frame (sample_move of the warp-level kernel)
__device__ __forceinline__ int pick_move(const DevConfig &cfg, const MoveSets &ms, int total, uint32_t rnd)
{
    if (total == 0) return cfg.A - 1;
    int t = int(__umulhi(rnd, uint32_t(total)));
    if (ms.any_far == 0) {
        // one-square moves only: the cell that holds move t is the last cell with at most t moves in the cells before it
        auto below = [&](int p) {
            const uint32_t low = (1u << p) - 1u;
            return __popc(ms.down & low) + __popc(ms.up & low) + __popc(ms.right & low) + __popc(ms.left & low);
        };
        int p = 0;
#pragma unroll
        for (int w = 8; w >= 1; w >>= 1)
            if (below(p + w) <= t) p += w;
        int r = t - below(p);
        // the cell's channels in ascending order: down 0 < up R-1 < right 2(R-1) < left 2(R-1)+C-1
        const int b1 = cfg.R - 1, b2 = 2 * b1, b3 = b2 + cfg.C - 1;
        const int d0 = int((ms.down >> p) & 1u), d1 = int((ms.up >> p) & 1u), d2 = int((ms.right >> p) & 1u);
        int ch = b3;
        if (r < d0) ch = 0;
        else if (r < d0 + d1) ch = b1;
        else if (r < d0 + d1 + d2) ch = b2;
        return p * cfg.A + ch;
    }
    int action = 0;
#pragma unroll 1
    for (int p = 0; p < cfg.N; ++p) {  // scouts on the board: walk the cells
        uint32_t w = cell_channels(cfg, ms, p);
        const int cnt = __popc(w);
        if (t < cnt) {
            for (int skip = t; skip > 0; --skip) w &= w - 1;
            action = p * cfg.A + __ffs(w) - 1;
            break;
        }
        t -= cnt;
    }
    return action;
}

// the 0/1 mask row [cell][channel] of a game: a 1 at every move (the row is zero on entry)
__device__ __forceinline__ void mark_row(const DevConfig &cfg, const MoveSets &ms, uint8_t *row)
{
    const int A = cfg.A, b1 = cfg.R - 1, b2 = 2 * b1, b3 = b2 + cfg.C - 1;
    for (uint32_t w = ms.down; w != 0; w &= w - 1) row[(__ffs(w) - 1) * A] = 1;
    for (uint32_t w = ms.up; w != 0; w &= w - 1) row[(__ffs(w) - 1) * A + b1] = 1;
    for (uint32_t w = ms.right; w != 0; w &= w - 1) row[(__ffs(w) - 1) * A + b2] = 1;
    for (uint32_t w = ms.left; w != 0; w &= w - 1) row[(__ffs(w) - 1) * A + b3] = 1;
    if (ms.any_far != 0) {
        const uint32_t far[8] = {ms.f0, ms.f1, ms.f2, ms.f3, ms.f4, ms.f5, ms.f6, ms.f7};
#pragma unroll
        for (int i = 0; i < 8; ++i)
            for (uint32_t w = far[i]; w != 0; w &= w - 1) {
                const int b = __ffs(w) - 1;
                row[(b & 15) * A + 2 * i + (b >> 4)] = 1;
            }
    }
}

// Observation tiles hold the background image permanently; per game the lanes first put the background back where the
// tile's previous game had entries (restore_tile, from a per-lane undo word) and then add the new game's entries
// (patch_tile, one pass of patch_obs of the warp-level kernel): lanes 0..N-1 their cell's one-hot / lake / still entries,
// lanes 16..19 the recent-move squares, lanes 20..27 the capture entries.  Undo word: cell lanes = four channel
// numbers (0 = none or channel 0: both restore to the zero background); the others = bit 31 valid | capture type << 16 |
// float offset, UNDO_NONE = nothing.
constexpr uint32_t UNDO_NONE = 0xffffffffu;

// Bytes of shared memory a 16-bit observation tile of `bytes` bytes takes: room to start it at the residue mod 16 its
// game's row has in the output tensor (0 or 8: rows are a multiple of 8 bytes, cells a multiple of 4).
__host__ __device__ inline int tile_slot(int bytes) { return bytes ? round16(bytes) + 16 : 0; }

// T: observation element, float or uint16_t (obs_value)
template <class T = float>
__device__ __forceinline__ void restore_tile(const DevConfig &cfg, T *tile, const ObsMap om, int lane, uint32_t undo)
{
    if (lane < cfg.N) {  // four unconditional stores: "no entry" is recorded as channel 0, whose background is zero too
        T *cell = tile + lane * om.channels;
        const T zero = obs_value<T>(cfg.unit_lut[0]);
#pragma unroll
        for (int k = 0; k < 4; ++k) cell[(undo >> (8 * k)) & 0xffu] = zero;
    } else if (lane >= 16 && undo != UNDO_NONE) {
        tile[undo & 0xffffu] = obs_value<T>(lane < 20 ? cfg.recent_lut[3] : cfg.cap_lut[((undo >> 16) & 15u) * 9]);
    }
}

template <class T = float>
__device__ __forceinline__ uint32_t patch_tile(const DevConfig &cfg, const uint8_t *stage, T *tile, const ObsMap om, int lane)
{
    const uint32_t info0 = *reinterpret_cast<const uint32_t *>(stage + 32), info1 = *reinterpret_cast<const uint32_t *>(stage + 36);
    const int me = (info1 >> 16) & 1, flip = me, CH = om.channels, N = cfg.N;
    const T one = obs_value<T>(cfg.unit_lut[1]);
    uint32_t undo = UNDO_NONE;
    if (lane < N) {
        const uint32_t b = stage[view(lane, flip, N)];
        T *cell = tile + lane * CH;
        uint32_t c0 = 0xff, c1 = 0xff, c2 = 0xff, c3 = 0xff;
        if (b & CELL_OBST) c0 = om.obstacle;
        const int rank = b & CELL_RANK;
        if (rank) {
            const int po = (b & CELL_REVEALED) ? rank : SP_UNKNOWN;
            const bool own = int((b >> 4) & 1) == me;
            if (own) c1 = om.own_true + rank - 1;
            else if (om.enemy_true >= 0) c1 = om.enemy_true + rank - 1;
            c2 = (own ? om.own_po : om.enemy_po) + po - 1;
            if (b & CELL_STILL) c3 = own ? om.own_still : om.enemy_still;
        }
        if (c0 != 0xff) cell[c0] = one;
        if (c1 != 0xff) cell[c1] = one;
        if (c2 != 0xff) cell[c2] = one;
        if (c3 != 0xff) cell[c3] = one;
        // undo word: the channels written, none = channel 0 (own_true's first plane: background zero, restore_tile)
        undo = (c0 == 0xff ? 0u : c0) | ((c1 == 0xff ? 0u : c1) << 8) | ((c2 == 0xff ? 0u : c2) << 16) | ((c3 == 0xff ? 0u : c3) << 24);
    } else if (lane >= 16 && lane < 20) {  // lanes 16/17 own from/to, 18/19 enemy from/to
        const int l = lane - 16, who = (l < 2) ? me : (me ^ 1);
        const uint32_t sq = who == 0 ? (info0 & 0xffffu) : (info0 >> 16);
        const int cell_abs = (l & 1) ? int(sq >> 8) : int(sq & 0xff);
        const int rcode = who == 0 ? int(info1 & 0xf) : int((info1 >> 4) & 0xf);
        const int code = (l & 1) ? -rcode : 1;
        if (cell_abs != NO_CELL) {
            const uint32_t off = uint32_t(view(cell_abs, flip, N) * CH + (l < 2 ? om.own_recent : om.enemy_recent));
            tile[off] = obs_value<T>(cfg.recent_lut[code + 3]);
            undo = 0x80000000u | off;
        }
    } else if (lane >= 20 && lane < 28) {
        const int e = lane - 20, ncap = (info1 >> 8) & 0xff;
        if (e < ncap) {
            const uint32_t ent = reinterpret_cast<const uint16_t *>(stage + 16)[e];
            const int cell_abs = ent & 0xff, owner = (ent >> 8) & 1, type0 = (ent >> 9) & 15, count = int(ent >> 13) + 1;
            const uint32_t off = uint32_t(view(cell_abs, flip, N) * CH + (owner == me ? om.own_cap : om.enemy_cap) + type0);
            tile[off] = obs_value<T>(cfg.cap_lut[type0 * 9 + count]);
            undo = 0x80000000u | (uint32_t(type0) << 16) | off;
        }
    }
    return undo;
}

}  // namespace toy
}  // namespace sx

