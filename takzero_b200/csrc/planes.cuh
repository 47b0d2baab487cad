// planes.cuh -- the f32 input planes of one position in shared memory (network/repr.rs:169-228), shared by the novelty
// hashes (nn.cu) and the RND estimator (rnd.cu).
#pragma once
#include "encode.cuh"
#include "rules.cuh"

// f32 input planes of one position (shared memory) straight to `out` [C][N][N], `game_repr` order: tz_encode_planes
// and the training batches.  The lanes own the squares; the indicator channels are the bits the fused network's
// first-layer producer encodes (enc::square_indicator_bits).
__device__ __forceinline__ void warp_encode_planes(const TzState* st, int n, int half_komi, float* out, int lane) {
    const int nn = n * n, ss = 2 * n + 3;
    const int me = st->to_move, other = me ^ 1;
    const TzBoards b = warp_boards(st, nn, lane);
    const int s0 = n == 3 ? 10 : n == 4 ? 15 : n == 5 ? 21 : 30;
    const int c0 = n >= 5 ? 1 : 0;
    const float my_stones = __fdiv_rn((float)st->stones[me], (float)s0);
    const float my_caps = c0 ? __fdiv_rn((float)st->caps[me], (float)c0) : 0.0f;
    const float op_stones = __fdiv_rn((float)st->stones[other], (float)s0);
    const float op_caps = c0 ? __fdiv_rn((float)st->caps[other], (float)c0) : 0.0f;
    const float fcd = __fsub_rn((float)(__popcll(b.flat[0]) - __popcll(b.flat[1])), __fdiv_rn((float)half_komi, 2.0f));
    const float fcd_sq = __fdiv_rn(fcd, (float)nn);
    const float side = me == 1 ? 1.0f : 0.0f;
    for (int sq = lane; sq < nn; sq += 32) {
        const uint64_t ones = enc::square_indicator_bits(st->stack[sq], st->height[sq], st->top[sq], me, n);
        float* o = out + sq;
        for (int c = 0; c < 2 * ss; c++) o[(size_t)c * nn] = (ones >> c) & 1ull ? 1.0f : 0.0f;
        const int base = 2 * ss;
        o[(size_t)(base + 0) * nn] = my_stones;
        o[(size_t)(base + 1) * nn] = my_caps;
        o[(size_t)(base + 2) * nn] = op_stones;
        o[(size_t)(base + 3) * nn] = op_caps;
        o[(size_t)(base + 4) * nn] = side;
        o[(size_t)(base + 5) * nn] = fcd_sq;
    }
}

// f32 input planes of one position into shared memory (x[plane * nn + square], `game_repr` order); the warp's
// lanes own the squares.  zero_colour leaves the "black to move" plane at 0 (SimHash, net6_simhash.rs:209-222).
__device__ __forceinline__ void warp_fill_planes(float* x, const TzState* st, int n, int half_komi, int lane,
                                                 bool zero_colour) {
    const int nn = n * n, ss = 2 * n + 3, C = 2 * (ss + 2) + 2;
    for (int i = lane; i < C * nn; i += 32) x[i] = 0.0f;
    __syncwarp();
    const int me = st->to_move, other = me ^ 1;
    const TzBoards b = warp_boards(st, nn, lane);
    const int s0 = n == 3 ? 10 : n == 4 ? 15 : n == 5 ? 21 : 30;
    const int c0 = n >= 5 ? 1 : 0;
    const float r0 = __fdiv_rn((float)st->stones[me], (float)s0);
    const float r1 = c0 ? __fdiv_rn((float)st->caps[me], (float)c0) : 0.0f;
    const float r2 = __fdiv_rn((float)st->stones[other], (float)s0);
    const float r3 = c0 ? __fdiv_rn((float)st->caps[other], (float)c0) : 0.0f;
    const float fcd = __fsub_rn((float)(__popcll(b.flat[0]) - __popcll(b.flat[1])), __fdiv_rn((float)half_komi, 2.0f));
    const float fcd_sq = __fdiv_rn(fcd, (float)nn);
    for (int sq = lane; sq < nn; sq += 32) {
        const int h = st->height[sq];
        if (h > 0) {
            const uint64_t stack = st->stack[sq];
            const int top_col = (int)((stack >> (h - 1)) & 1ull);
            x[(st->top[sq] + (top_col != me ? ss : 0)) * nn + sq] = 1.0f;
            for (int i = 0; i < ss - 3 && h - 2 - i >= 0; i++) {
                const int col = (int)((stack >> (h - 2 - i)) & 1ull);
                x[(3 + i + (col != me ? ss : 0)) * nn + sq] = 1.0f;
            }
        }
        const int base = 2 * ss;
        x[(base + 0) * nn + sq] = r0;
        x[(base + 1) * nn + sq] = r1;
        x[(base + 2) * nn + sq] = r2;
        x[(base + 3) * nn + sq] = r3;
        if (!zero_colour && me == 1) x[(base + 4) * nn + sq] = 1.0f;
        x[(base + 5) * nn + sq] = fcd_sq;
    }
    __syncwarp();
}

