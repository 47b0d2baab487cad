// rules.cuh -- warp-per-game Tak rules on a shared-memory TzState (sm_100a).
//
// Replaces, for the hot path, what the reference gets from the crate fast-tak 0.4.1
// through takzero/src/search/env.rs:39-59 (`possible_moves`, `play`, `result`).
// One warp owns one game; lanes own squares (sq = row*N + col; lanes 0..3 own a
// second square for N = 6).  Bitboards are built with warp ballots.
#pragma once
#include "common.cuh"

#define FULL_MASK 0xffffffffu

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// ---- load / store -------------------------------------------------------------

__device__ __forceinline__ void warp_load_state(TzState* dst, const TzState* src, int lane) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    if (lane < 24) d[lane] = s[lane];
    __syncwarp();
}

__device__ __forceinline__ void warp_store_state(TzState* dst, const TzState* src, int lane) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
    uint4* d = reinterpret_cast<uint4*>(dst);
    __syncwarp();
    if (lane < 24) d[lane] = s[lane];
}

// ---- bitboards -------------------------------------------------------------------

struct TzBoards {
    uint64_t occ, road[2], flat[2], wall, cap;
};

__device__ __forceinline__ TzBoards warp_boards(const TzState* s, int nn, int lane) {
    TzBoards b;
    uint32_t occ[2], r0[2], r1[2], f0[2], f1[2], w[2], c[2];
#pragma unroll
    for (int slot = 0; slot < 2; slot++) {
        const int sq = lane + 32 * slot;
        int h = 0, t = 0, col = 0;
        if (sq < nn) {
            h = s->height[sq];
            t = s->top[sq];
            if (h > 0) col = (int)((s->stack[sq] >> (h - 1)) & 1ull);
        }
        const bool on = h > 0;
        occ[slot] = __ballot_sync(FULL_MASK, on);
        r0[slot] = __ballot_sync(FULL_MASK, on && t != TZ_WALL && col == 0);
        r1[slot] = __ballot_sync(FULL_MASK, on && t != TZ_WALL && col == 1);
        f0[slot] = __ballot_sync(FULL_MASK, on && t == TZ_FLAT && col == 0);
        f1[slot] = __ballot_sync(FULL_MASK, on && t == TZ_FLAT && col == 1);
        w[slot] = __ballot_sync(FULL_MASK, on && t == TZ_WALL);
        c[slot] = __ballot_sync(FULL_MASK, on && t == TZ_CAP);
    }
    b.occ = occ[0] | ((uint64_t)occ[1] << 32);
    b.road[0] = r0[0] | ((uint64_t)r0[1] << 32);
    b.road[1] = r1[0] | ((uint64_t)r1[1] << 32);
    b.flat[0] = f0[0] | ((uint64_t)f0[1] << 32);
    b.flat[1] = f1[0] | ((uint64_t)f1[1] << 32);
    b.wall = w[0] | ((uint64_t)w[1] << 32);
    b.cap = c[0] | ((uint64_t)c[1] << 32);
    return b;
}

__device__ __forceinline__ uint64_t row_mask(int n, int row) { return ((1ull << n) - 1) << (row * n); }
__device__ __forceinline__ uint64_t col_mask(int n, int col) {
    uint64_t m = 0;
    for (int r = 0; r < n; r++) m |= 1ull << (r * n + col);
    return m;
}

// flood fill from `from` through `road`, true when `to` is reached
__device__ __forceinline__ bool bb_connects(uint64_t road, uint64_t from, uint64_t to, int n,
                                            uint64_t not_col0, uint64_t not_colN) {
    uint64_t reach = road & from;
    while (reach) {
        if (reach & to) return true;
        uint64_t grow = (reach << n) | (reach >> n) | ((reach << 1) & not_col0) | ((reach >> 1) & not_colN);
        uint64_t next = (reach | grow) & road;
        if (next == reach) break;
        reach = next;
    }
    return false;
}

// fast-tak's `Game::result` as consumed by env.rs:47-59 and target.rs:226-230: road for the player who
// just moved first, then the other player, then flat count (komi) when the board is full or a player is
// out of pieces, then the reversible-ply draw.
// Returns 0 ongoing, 1 white road, 2 black road, 3 white flat win, 4 black flat win, 5 draw.
__device__ __forceinline__ int warp_game_result(const TzState* s, int n, int half_komi, int rev_limit, int lane) {
    const int nn = n * n;
    const TzBoards b = warp_boards(s, nn, lane);
    const uint64_t c0 = col_mask(n, 0), cN = col_mask(n, n - 1);
    bool mine = false;
    if (lane < 4) {
        const int color = lane >> 1;
        if (lane & 1)
            mine = bb_connects(b.road[color], c0, cN, n, ~c0, ~cN);
        else
            mine = bb_connects(b.road[color], row_mask(n, 0), row_mask(n, n - 1), n, ~c0, ~cN);
    }
    const uint32_t roads = __ballot_sync(FULL_MASK, mine);
    const bool road_w = roads & 3u, road_b = roads & 12u;
    const int to_move = s->to_move, mover = to_move ^ 1;
    const bool road_mover = mover == 0 ? road_w : road_b;
    const bool road_other = mover == 0 ? road_b : road_w;
    if (road_mover) return 1 + mover;
    if (road_other) return 1 + to_move;
    const bool full = __popcll(b.occ) == nn;
    const bool w_out = s->stones[0] == 0 && s->caps[0] == 0;
    const bool b_out = s->stones[1] == 0 && s->caps[1] == 0;
    if (full || w_out || b_out) {
        const int score2 = 2 * (__popcll(b.flat[0]) - __popcll(b.flat[1])) - half_komi;
        return score2 > 0 ? 3 : (score2 < 0 ? 4 : 5);
    }
    if ((int)s->reversible_plies >= rev_limit) return 5;
    return 0;
}

// `Environment::terminal` (env.rs:47-59): the result relative to the side to move
__device__ __forceinline__ int warp_terminal(const TzState* s, int n, int half_komi, int rev_limit, int lane) {
    const int r = warp_game_result(s, n, half_komi, rev_limit, lane);
    if (r == 0) return TZ_T_NONE;
    if (r == 5) return TZ_T_DRAW;
    const int winner = (r == 1 || r == 3) ? 0 : 1;
    return winner == (int)s->to_move ? TZ_T_WIN : TZ_T_LOSS;
}

// ---- move generation -----------------------------------------------------------

__device__ __forceinline__ int tz_binom(int n, int k) {
    if (k < 0 || k > n) return 0;
    uint32_t row;
    switch (n) {
        case 0: row = 0x1; break;
        case 1: row = 0x11; break;
        case 2: row = 0x121; break;
        case 3: row = 0x1331; break;
        case 4: row = 0x14641; break;
        default: row = 0x15AA51; break;
    }
    return (row >> (4 * k)) & 0xF;
}

__device__ __forceinline__ uint16_t tz_mk_move(int row, int col, int kind, int pat) {
    return (uint16_t)(col | (row << 3) | (kind << 6) | (pat << 8));
}

// number of legal drop sequences for `c` carried pieces, `reach` free squares and an
// optional capstone flattening of a wall on square reach+1
// (compositions of c into at most `reach` parts = sum_{j < min(reach, c)} C(c-1, j): partial sums of the binomial
// rows, one byte per limit, looked up instead of added up -- this is the hottest arithmetic of k_select)
__device__ __forceinline__ int spread_count(int c, int reach, bool smash) {
    const int lim = reach < c ? reach : c;
    unsigned long long sums;  // byte (lim - 1) = sum_{j < lim} C(c - 1, j)
    switch (c) {
        case 1: sums = 0x01ull; break;
        case 2: sums = 0x0201ull; break;
        case 3: sums = 0x040301ull; break;
        case 4: sums = 0x08070401ull; break;
        case 5: sums = 0x100f0b0501ull; break;
        default: sums = 0x201f1a100601ull; break;
    }
    int cnt = lim > 0 ? (int)((sums >> (8 * (lim - 1))) & 0xffull) : 0;
    if (smash && reach + 1 <= c) cnt += reach == 0 ? (c == 1) : tz_binom(c - 2, reach - 1);
    return cnt;
}

struct SquareDirs {
    int free_run[4];   // consecutive squares a spread may enter
    bool wall_next[4]; // the square after them holds a wall
};

__device__ __forceinline__ void square_dirs(const TzState* s, int n, int row, int col, SquareDirs& d) {
    const int dr[4] = {1, -1, 0, 0}, dc[4] = {0, 0, -1, 1};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        int r = row, c = col, run = 0;
        bool wall = false;
        for (int step = 1; step < n; step++) {
            r += dr[k];
            c += dc[k];
            if (r < 0 || r >= n || c < 0 || c >= n) break;
            const int t = r * n + c;
            if (s->height[t] > 0 && s->top[t] != TZ_FLAT) {
                wall = s->top[t] == TZ_WALL;
                break;
            }
            run = step;
        }
        d.free_run[k] = run;
        d.wall_next[k] = wall;
    }
}

// Legal moves in fast-tak order (SURVEY App. B.1, pinned by runs/*.txt): squares
// file-major, placements flat/wall/cap, spreads carry-major x (+,-,<,>) x descending
// lexicographic drops.  Writes u16 moves to `out` (shared memory) and returns the
// count (or -1 when more than TZ_MAX_MOVES).  Warp-convergent.  `ranges` (optional, global memory, 36 entries indexed by
// square = row * N + col) receives for every square the index of its first move | its move count << 16: the moves that
// start on one square are contiguous, which is what the policy convolution's epilogue gathers by (conv_tcgen05.cuh).
__device__ __forceinline__ int warp_movegen(const TzState* s, int n, uint16_t* out, int lane, uint32_t* ranges = nullptr) {
    const int nn = n * n;
    const int me = s->to_move;
    const bool opening = s->ply < 2;
    const bool can_stone = s->stones[me] > 0, can_cap = s->caps[me] > 0;
    int cnt[2] = {0, 0};
    uint32_t dirs[2] = {0, 0};  // per direction: free run (3 bits) | wall behind it << 3, kept for pass 2
    // pass 1: per-square counts, squares indexed in generation order k = col*n + row
#pragma unroll
    for (int slot = 0; slot < 2; slot++) {
        const int k = lane + 32 * slot;
        if (k >= nn) continue;
        const int col = k / n, row = k % n, sq = row * n + col;
        const int h = s->height[sq];
        if (h == 0) {
            cnt[slot] = opening ? 1 : (can_stone ? 2 : 0) + (can_cap ? 1 : 0);
        } else if (!opening && (int)((s->stack[sq] >> (h - 1)) & 1ull) == me) {
            SquareDirs d;
            square_dirs(s, n, row, col, d);
#pragma unroll
            for (int k2 = 0; k2 < 4; k2++) dirs[slot] |= (uint32_t)(d.free_run[k2] | (d.wall_next[k2] ? 8 : 0)) << (4 * k2);
            const bool is_cap = s->top[sq] == TZ_CAP;
            const int maxc = h < n ? h : n;
            int c_total = 0;
            for (int c = 1; c <= maxc; c++)
#pragma unroll
                for (int k2 = 0; k2 < 4; k2++) {
                    const int reach = d.free_run[k2] < c ? d.free_run[k2] : c;
                    const bool smash = is_cap && d.wall_next[k2] && d.free_run[k2] < c;
                    c_total += spread_count(c, reach, smash);
                }
            cnt[slot] = c_total;
        }
    }
    // exclusive scan in generation order (slot 0 lanes first, then slot 1)
    int inc0 = cnt[0];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(FULL_MASK, inc0, o);
        if (lane >= o) inc0 += v;
    }
    const int total0 = __shfl_sync(FULL_MASK, inc0, 31);
    int inc1 = cnt[1];
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        const int v = __shfl_up_sync(FULL_MASK, inc1, o);
        if (lane >= o) inc1 += v;
    }
    const int total = total0 + __shfl_sync(FULL_MASK, inc1, 7);
    if (total > TZ_MAX_MOVES) return -1;
    int off[2] = {inc0 - cnt[0], total0 + inc1 - cnt[1]};
    if (ranges != nullptr) {
#pragma unroll
        for (int slot = 0; slot < 2; slot++) {
            const int k = lane + 32 * slot;
            if (k < nn) ranges[(k % n) * n + k / n] = (uint32_t)off[slot] | ((uint32_t)cnt[slot] << 16);
        }
    }
    // pass 2: each lane writes its squares' moves
#pragma unroll
    for (int slot = 0; slot < 2; slot++) {
        const int k = lane + 32 * slot;
        if (k >= nn || cnt[slot] == 0) continue;
        const int col = k / n, row = k % n, sq = row * n + col;
        int o = off[slot];
        const int h = s->height[sq];
        if (h == 0) {
            if (opening) {
                out[o++] = tz_mk_move(row, col, TZ_FLAT, 0);
            } else {
                if (can_stone) {
                    out[o++] = tz_mk_move(row, col, TZ_FLAT, 0);
                    out[o++] = tz_mk_move(row, col, TZ_WALL, 0);
                }
                if (can_cap) out[o++] = tz_mk_move(row, col, TZ_CAP, 0);
            }
        } else {
            const bool is_cap = s->top[sq] == TZ_CAP;
            const int maxc = h < n ? h : n;
            for (int c = 1; c <= maxc; c++)
                for (int k2 = 0; k2 < 4; k2++) {
                    const int run = (int)((dirs[slot] >> (4 * k2)) & 7u);
                    const bool wall = (dirs[slot] >> (4 * k2 + 3)) & 1u;
                    const int reach = run < c ? run : c;
                    const bool smash = is_cap && wall && run < c;
                    if (reach == 0 && !smash) continue;
                    const bool all = reach >= c;  // every drop sequence fits: no per-pattern test
                    for (int rev = 1 << (c - 1); rev < (1 << c); rev++) {
                        if (!all) {
                            const int parts = __popc(rev);
                            if (!(parts <= reach || (smash && parts == reach + 1 && (rev & 1)))) continue;
                        }
                        // pattern byte: bit (8-c+i) = bit (c-1-i) of rev
                        const int pat = (int)(__brev((unsigned)rev) >> (32 - c)) << (8 - c);
                        out[o++] = tz_mk_move(row, col, k2, pat);
                    }
                }
        }
    }
    __syncwarp();
    return total;
}

// ---- apply ---------------------------------------------------------------------

// fast-tak `Game::play` for a move already known to be legal (env.rs:43-45).  Lane 0
// mutates the shared-memory state; returns false on a malformed move.
__device__ __forceinline__ bool warp_apply(TzState* s, int n, uint16_t m, int lane) {
    bool ok = true;
    if (lane == 0) {
        const int col = m & 7, row = (m >> 3) & 7, kind = (m >> 6) & 3, pat = m >> 8;
        const int me = s->to_move;
        const int sq = row * n + col;
        if (row >= n || col >= n) {
            ok = false;
        } else if (pat == 0) {
            const int color = s->ply < 2 ? (me ^ 1) : me;
            if (s->height[sq] != 0 || kind > TZ_CAP || (s->ply < 2 && kind != TZ_FLAT)) ok = false;
            if (kind == TZ_CAP) {
                if (s->caps[color] == 0) ok = false;
                else s->caps[color]--;
            } else {
                if (s->stones[color] == 0) ok = false;
                else s->stones[color]--;
            }
            s->stack[sq] = (uint64_t)color;
            s->height[sq] = 1;
            s->top[sq] = (uint8_t)kind;
            s->reversible_plies = 0;
        } else {
            const int drow = (kind == 0) - (kind == 1), dcol = (kind == 3) - (kind == 2);
            const int h = s->height[sq];
            const int c = 8 - (__ffs(pat) - 1);
            if (s->ply < 2 || h == 0 || c > h || c > n || (int)((s->stack[sq] >> (h - 1)) & 1ull) != me) {
                ok = false;
            } else {
                const uint64_t carried = (s->stack[sq] >> (h - c)) & ((1ull << c) - 1);
                const int toptype = s->top[sq];
                s->height[sq] = (uint8_t)(h - c);
                s->stack[sq] &= (1ull << (h - c)) - 1;
                s->top[sq] = TZ_FLAT;
                int r = row, cc = col, pos = sq;
                bool smashed = false;
                for (int i = 0; i < c; i++) {
                    if ((pat >> (8 - c + i)) & 1) {
                        r += drow;
                        cc += dcol;
                        if (r < 0 || r >= n || cc < 0 || cc >= n) {
                            ok = false;
                            break;
                        }
                        pos = r * n + cc;
                        if (s->height[pos] > 0 && s->top[pos] == TZ_WALL) smashed = true;
                    }
                    s->stack[pos] |= ((carried >> i) & 1ull) << s->height[pos];
                    s->height[pos]++;
                    s->top[pos] = TZ_FLAT;
                }
                s->top[pos] = (uint8_t)toptype;
                s->reversible_plies = smashed ? 0 : (uint16_t)(s->reversible_plies + 1);
            }
        }
        s->ply++;
        s->to_move ^= 1;
    }
    __syncwarp();
    return __shfl_sync(FULL_MASK, ok ? 1 : 0, 0) != 0;
}

// ---- hash (shared with oracle/tak_rules.c `tk_state_hash`) -----------------------

__host__ __device__ __forceinline__ uint64_t tz_mix64(uint64_t x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdULL;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ULL;
    x ^= x >> 33;
    return x;
}

__device__ __forceinline__ uint64_t warp_state_hash(const TzState* s, int nn, int lane) {
    uint64_t acc = 0;
    for (int sq = lane; sq < nn; sq += 32) {
        const uint64_t hh = s->height[sq];
        const uint64_t tt = hh ? s->top[sq] : 0;
        acc += tz_mix64(s->stack[sq] * 0x100000001b3ULL + (hh << 8) + (tt << 16) + ((uint64_t)(sq + 1) << 24));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(FULL_MASK, acc, o);
    return tz_mix64(acc + (0x9e3779b97f4a7c15ULL ^ (uint64_t)s->to_move));
}

// the library's counter-based generator (stated at tz_training_batch in the header)
__device__ __forceinline__ uint64_t rng_hash(uint64_t seed, uint64_t a, uint64_t b, uint64_t c) {
    uint64_t h = tz_mix64(seed ^ 0x9e3779b97f4a7c15ULL);
    h = tz_mix64(h ^ (a * 0xbf58476d1ce4e5b9ULL));
    h = tz_mix64(h ^ (b * 0x94d049bb133111ebULL));
    return tz_mix64(h ^ (c * 0xd6e8feb86659fd93ULL));
}

// ---- board symmetries of the training batches (tz_training_batch, tz_update_counts_buffer) -----------

// symmetry t of the board: bit 0 mirrors the column, bit 1 the row, bit 2 swaps them, in this order
__device__ __forceinline__ void sym_square(int t, int n, int* row, int* col) {
    if (t & 1) *col = n - 1 - *col;
    if (t & 2) *row = n - 1 - *row;
    if (t & 4) {
        const int tmp = *col;
        *col = *row;
        *row = tmp;
    }
}

// example b of a batch: target `index` (counted from the oldest kept one of `size`) under symmetry `t`, explicit or
// drawn as the header states at tz_training_batch
__device__ __forceinline__ void batch_example(const unsigned long long* indices, const int* symmetry, int augment,
                                              unsigned long long seed, unsigned long long size, int b,
                                              unsigned long long* index, int* t) {
    *index = indices ? indices[b] : __umul64hi(rng_hash(seed, (uint64_t)b, 0, 0), size);
    *t = symmetry ? symmetry[b] : augment ? (int)(rng_hash(seed, (uint64_t)b, 1, 0) & 7) : 0;
}

// dst = src under symmetry t (shared memory, one warp): the squares move, reserves, side to move and plies are kept
__device__ __forceinline__ void warp_symmetric_state(TzState* dst, const TzState* src, int t, int n, int lane) {
    warp_load_state(dst, src, lane);
    const int nn = n * n;
    for (int sq = lane; sq < nn; sq += 32) {
        int row = sq / n, col = sq - row * n;
        sym_square(t, n, &row, &col);
        const int to = row * n + col;
        dst->stack[to] = src->stack[sq];
        dst->height[to] = src->height[sq];
        dst->top[to] = src->top[sq];
    }
    __syncwarp();
}
